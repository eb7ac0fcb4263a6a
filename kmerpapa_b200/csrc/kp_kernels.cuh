// kp_kernels.cuh — sm_100a kernels of the pattern-partition DP.
//
// Work decomposition (geometry in kp_tables.h, rationale in DESIGN.md):
//
//  K3+K4  kp_dp_rows_kernel   the min-plus recurrence with the float64 self-score fused in, lazily.
//      One WARP owns one tile at a time, one LANE owns one row of it, and the r0 (<= 15) sub-patterns of
//      the register position of that row live in registers.  No block-wide barrier in steady state.
//      Per tile:
//        phase D  (single DP) stream the two child tiles of every HIGH-position split for all rows, 32
//                 consecutive rows at a time, coalesced 16-byte loads, one flattened two-deep software
//                 pipeline; the running minimum of each row is parked in shared memory.
//        rounds   rows are visited in a precomputed schedule (<= 32 rows whose children are complete):
//                 running minimum over the CROSS-row splits from the tile's finished rows in shared memory;
//                 counts of the row from the tile's base k-mers by subset sums;
//                 SCORE FILTER: a float32 estimate of every self-score with a rigorous error margin; a
//                 pattern whose estimate minus margin already exceeds its best split so far can never be
//                 kept whole (later in-register splits only lower the best split), so its exact score is
//                 never needed;
//                 SCORE for the remaining patterns only, in a rolled loop (the code exists once): a fast float64
//                 evaluation with a rigorous error bound (kp_self_score_fast) decides RN_f32(s) and the "rounded up"
//                 bit for all but about one score in 10^5, which take the glibc-exact path (kp_math.cuh); both are kept because
//                 the reference's float64 compare  s < (double)best  is exactly
//                 sf < best || (sf == best && rounded_up), and the value it stores on a win is sf;
//                 in-register splits of the register position interleaved with that compare, fully
//                 unrolled; one coalesced 16-byte store per group, one 16-bit "kept whole" mask per row.
//      The kernel only keeps the minimum (fminf); which split won is re-derived by the backtrack from the
//      stored scores (first split in scan order that reproduces the minimum).
//
//  CV job = the same kernel on the TRAIN counts (total - held-out).  The reference also carries the held-out
//      loss of every pattern's best partition, but only reads it at the general pattern; that value is the
//      float32 sum, along the optimal partition tree, of the leaves' held-out losses, so it is computed
//      after the DP from the backtracked tree (kp_cv_leaf_kernel + a host reduction in tree order).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "kp_math.cuh"
#include "kp_tables.h"

// Tiles in flight per SM.  Warps are allocated four at a time, so 13-16 warps leave 128 registers per thread, 12 leave
// 170: measured 14 warps / 128 registers (spills, tight scheduling) 27.1 ms, 12 warps / 161 registers 25.4 ms, 10: 26.6,
// 8: 29.3 (one 9-mer DP, tools/ab_libs.sh).
#ifndef KP_MAX_WARPS
#define KP_MAX_WARPS 12
#endif
#define KP_DP_BOUNDS __launch_bounds__(KP_MAX_WARPS * 32, 1)
#ifndef KP_PIPE_DEPTH
#define KP_PIPE_DEPTH 2      // register stages of the child-tile stream (3 needs <= 13 warps for its registers)
#endif
// Experimental variants of the child-tile stream measured in round 2 and found not to help (profiles/r02_l2_experiments.txt):
// L2 evict-first policy loads for the top positions' children (KP_EVICT_TOP), prefetch of the top positions' splits only
// (KP_PF_TOP), bulk L2 prefetch (KP_PF_BULK).  Compiled in only with -DKP_EXPERIMENTS=1: they lengthen the hot loop's code.
#ifndef KP_EXPERIMENTS
#define KP_EXPERIMENTS 0
#endif
#ifndef KP_PF_DIST
#define KP_PF_DIST 2         // L2 prefetch distance of the child-tile stream, in (32 rows x 1 split) steps
#endif

template <bool WIDE> struct KpCnt { typedef unsigned int type; };
template <> struct KpCnt<true> { typedef unsigned long long type; };

__device__ __forceinline__ double kp_cnt2d(unsigned int x) { return __uint2double_rn(x); }
__device__ __forceinline__ double kp_cnt2d(unsigned long long x) { return __ull2double_rn(x); }

// level >= 1 self-score (w_numba.py:56-61 / _CV.py:60-70), templated on the on-chip count width.
// log p takes the table path and log(1-p) the near-1 polynomial for every realistic rate; anything else
// (p >= 0.9375, p == 0, 1-p == 1, ...) goes through the out-of-line generic log.  No branches on M, U:
// the unselected products may be NaN/inf and are discarded by the selects.
template <typename C>
__device__ __forceinline__ double kp_self_score_t(C M, C U, double alpha, double beta, double penalty,
                                                  const double2 *tab, const KpLogK &K, double &logp, double &log1mp)
{
    double Md = kp_cnt2d(M), Ud = kp_cnt2d(U);
    double p = __ddiv_rn(KP_ADD(Md, alpha), KP_ADD(KP_ADD(kp_cnt2d((C)(M + U)), alpha), beta));
    double q = KP_SUB(1.0, p);
    int phi = __double2hiint(p), qhi = __double2hiint(q), qlo = __double2loint(q);
    if (kp_log_is_plain(phi) && !kp_log_is_near1(phi)) logp = kp_log_main(phi, __double2loint(p), tab, K);
    else logp = kp_log_slow(p, tab);
    if (kp_log_is_near1(qhi) && !(qhi == 0x3ff00000 && qlo == 0)) log1mp = kp_log_near1(q, K);
    else log1mp = kp_log_slow(q, tab);
    double s1 = KP_ADD(penalty, KP_MUL(KP_MUL(-2.0, Md), logp));
    double s = M > 0 ? s1 : penalty;
    double s2 = KP_ADD(s, KP_MUL(KP_MUL(-2.0, Ud), log1mp));
    return U > 0 ? s2 : s;
}

// out-of-line copy of the exact score: after kp_self_score_fast it is the rare path, and a call keeps its registers
// (the glibc-exact log needs a dozen live doubles) out of the hot loop
template <typename C>
__device__ __noinline__ double kp_self_score_exact_nl(C M, C U, double alpha, double beta, double penalty, const double2 *tab)
{
    const KpLogK K = kp_logk_load();
    double lp, l1;
    return kp_self_score_t<C>(M, U, alpha, beta, penalty, tab, K, lp, l1);
}

// FAST self-score with a rigorous error bound.  What the DP needs from the float64 score s of the reference
// (w_numba.py:56-64) is only  sf = RN_f32(s)  and the bit  (double)sf > s.  Both follow from ANY float64 approximation
// s~ with |s~ - s| <= eps unless s~ lies within eps of a float32 rounding boundary or of sf itself, which happens for
// about one score in 10^5; only those take the glibc-exact path.  s~ costs a third of the exact score: the quotient by
// a reciprocal seed and two Newton steps instead of the IEEE division, log p by glibc's table and polynomial without the
// hi/lo compensation, log(1-p) by a plain Horner evaluation of glibc's near-1 polynomial (five terms below 2^-8).
// Error budget (pen >= 0, 2^-1000 < p < 2^-4, so q = 1 - p > 0.9375 and |ln p| > 2.7; a = pen + t1 + t2 with
// t1 = -2 M ln p >= 0, t2 = -2 U ln q >= 0):
//   quotient        |p~ - p| <= 1.2 * 2^-50 p                 -> 2M * 1.2 * 2^-50 <= 2^-51 t1;  via q: 2U * 1.3 * 2^-50 p <= 2^-49 t2
//   rounding of q   |q~ - q| <= 2^-53 more, / q               -> 2U * 1.07 * 2^-53 <= 2^-51 (M + U)      [not relative to t2]
//   logs            this approximation <= 2^-50 relative, glibc's own < 1 ulp of the true log     -> 2^-49 (t1 + t2)
//   mul / add       four roundings in each sequence                                                -> 2^-50 a
//   total           < 2^-48 a + 2^-51 (M + U);   the bound used is  eps = 2^-46 a + 2^-49 (M + U).
// Returns false when the arguments are outside the window above (the caller then takes the exact path).
#ifndef KP_FAST_INLINE
#define KP_FAST_INLINE __forceinline__
#endif
// st (test hook only): receives s~; the DP kernels pass nothing and the store is compiled out.
template <typename C>
__device__ KP_FAST_INLINE bool kp_self_score_fast(C M, C U, double alpha, double beta, double penalty, const double2 *tab,
                                                   const KpLogK &K, float &sf, bool &rup, double *st = nullptr)
{
    const double Md = kp_cnt2d(M), Ud = kp_cnt2d(U), Sd = kp_cnt2d((C)(M + U));
    const double num = KP_ADD(Md, alpha), den = KP_ADD(KP_ADD(Sd, alpha), beta);
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(den));
    double e = KP_FMA(-den, r, 1.0);
    r = KP_FMA(r, e, r);
    e = KP_FMA(-den, r, 1.0);
    r = KP_FMA(r, e, r);
    const double p = KP_MUL(num, r);
    const int phi = __double2hiint(p), dhi = __double2hiint(den);
    // 2^-1000 <= p < 2^-4, 2^-500 <= den < 2^500 (the reciprocal seed flushes subnormals), pen >= 0
    bool ok = (unsigned)(phi - 0x01700000) < (unsigned)(0x3fb00000 - 0x01700000) &&
              (unsigned)(dhi - 0x20b00000) < (unsigned)(0x5f300000 - 0x20b00000) && penalty >= 0.0;
    // log p~
    const double *A = kpc_logA;
    const unsigned thi = (unsigned)phi - 0x3fe60000u;
    const int i = (int)((thi >> 13) & 127u);
    const int k = (int)thi >> 20;
    const double z = __hiloint2double(phi - (int)(thi & 0xfff00000u), __double2loint(p));
    const double2 t = tab[i];
    const double kd = (double)k;
    const double rr = KP_FMA(z, t.x, -1.0);
    const double r2 = KP_MUL(rr, rr);
    const double w = KP_FMA(kd, KP_LOG_LN2HI, t.y);
    double q1 = KP_FMA(rr, A[4], K.a3);
    const double q5 = KP_FMA(rr, A[2], K.a1);
    q1 = KP_FMA(q1, r2, q5);
    double lo = KP_FMA(kd, KP_LOG_LN2LO, rr);
    lo = KP_FMA(r2, A[0], lo);
    lo = KP_FMA(KP_MUL(rr, r2), q1, lo);
    const double logp = KP_ADD(w, lo);
    // log q~, q~ = 1 - p~ in (0.9375, 1]: ln(1 + x) = x + x^2 (B0 + x (B1 + ...)), x = q~ - 1 exactly
    const double *B = kpc_logB;
    const double x = KP_SUB(KP_SUB(1.0, p), 1.0);
    const double x2 = KP_MUL(x, x);
    double y;
    if (phi < 0x3f700000) {   // p < 2^-8: the terms beyond x^6 are below 2^-50 |x|
        y = KP_FMA(x, B[4], B[3]);
        y = KP_FMA(y, x, B[2]);
        y = KP_FMA(y, x, K.b1);
        y = KP_FMA(y, x, -0.5);
    } else {
        y = KP_FMA(x, B[10], B[9]);
        y = KP_FMA(y, x, B[8]);
        y = KP_FMA(y, x, K.b7);
        y = KP_FMA(y, x, B[6]);
        y = KP_FMA(y, x, B[5]);
        y = KP_FMA(y, x, K.b4);
        y = KP_FMA(y, x, B[3]);
        y = KP_FMA(y, x, B[2]);
        y = KP_FMA(y, x, K.b1);
        y = KP_FMA(y, x, -0.5);
    }
    const double logq = KP_FMA(x2, y, x);
    const double t1 = KP_MUL(KP_MUL(-2.0, Md), logp), t2 = KP_MUL(KP_MUL(-2.0, Ud), logq);
    double sa = M > 0 ? KP_ADD(penalty, t1) : penalty;
    sa = U > 0 ? KP_ADD(sa, t2) : sa;
    const double eps = KP_FMA(sa, 0x1p-46, KP_MUL(Sd, 0x1p-49));   // pen >= 0: sa = pen + t1 + t2 = a
    const double slo = KP_SUB(sa, eps), shi = KP_ADD(sa, eps);
    const float flo = __double2float_rn(slo), fhi = __double2float_rn(shi);
    const double fd = (double)flo;
    sf = flo;
    rup = fd > shi;
    if (st) *st = sa;
    ok = ok && flo == fhi && (fd > shi || fd < slo) && sa < 0x1p120;   // NaN / inf / ambiguous: exact path
    return ok;
}

// held-out -2 log-lik of a pattern kept whole (_CV.py:73-78), branch-free
template <typename C>
__device__ __forceinline__ double kp_test_ll_t(C Mt, C Ut, double logp, double log1mp)
{
    double t1 = KP_ADD(0.0, KP_MUL(KP_MUL(-2.0, kp_cnt2d(Mt)), logp));
    double t = Mt > 0 ? t1 : 0.0;
    double t2 = KP_ADD(t, KP_MUL(KP_MUL(-2.0, kp_cnt2d(Ut)), log1mp));
    return Ut > 0 ? t2 : t;
}

// subset sum of per-base counts for a compile-time base mask
template <int BM, int NB, typename C>
__device__ __forceinline__ C kp_sum_bases(const C *x)
{
    C s = 0;
#pragma unroll
    for (int b = 0; b < NB; b++)
        if ((BM >> b) & 1) s += x[b];
    return s;
}

// digit -> covered base digits of the register position (digit space), per radix
template <int R0> __host__ __device__ constexpr int kp_bm_c(int d)
{
    return R0 == 15 ? (d == 0 ? 1 : d == 1 ? 2 : d == 2 ? 4 : d == 3 ? 8 : d == 4 ? 5 : d == 5 ? 10 : d == 6 ? 6 : d == 7 ? 9 :
                       d == 8 ? 12 : d == 9 ? 3 : d == 10 ? 14 : d == 11 ? 13 : d == 12 ? 11 : d == 13 ? 7 : d == 14 ? 15 : 0)
         : R0 == 7 ? (d == 0 ? 1 : d == 1 ? 2 : d == 2 ? 4 : d == 3 ? 3 : d == 4 ? 5 : d == 5 ? 6 : d == 6 ? 7 : 0)
         : R0 == 3 ? (d == 0 ? 1 : d == 1 ? 2 : d == 2 ? 3 : 0)
         : (d == 0 ? 1 : 0);
}

// level-0 scores are rare (k-mers only): keep them out of line
__device__ __noinline__ double kp_leaf_score_nl(unsigned long long M, unsigned long long U, double alpha, double beta,
                                                double penalty, const double2 *tab)
{
    return kp_leaf_score(M, U, alpha, beta, penalty, tab);
}
__device__ __noinline__ void kp_leaf_cv_nl(unsigned long long Mtr, unsigned long long Utr, unsigned long long Mte,
                                           unsigned long long Ute, double alpha, double beta, double penalty,
                                           const double2 *tab, double *train, double *test)
{
    double a, b;
    kp_leaf_cv(Mtr, Utr, Mte, Ute, alpha, beta, penalty, tab, a, b);
    *train = a;
    *test = b;
}

// digit -> covered base digits of the register position (digit space), run-time index (exact-score loop)
__constant__ uint8_t kpc_bm1[4] = {1, 0, 0, 0};
__constant__ uint8_t kpc_bm3[4] = {1, 2, 3, 0};
__constant__ uint8_t kpc_bm7[8] = {1, 2, 4, 3, 5, 6, 7, 0};
__constant__ uint8_t kpc_bm15[16] = {1, 2, 4, 8, 5, 10, 6, 9, 12, 3, 14, 13, 11, 7, 15, 0};
template <int R0> __device__ __forceinline__ unsigned kp_bm(int d)
{
    return R0 == 15 ? kpc_bm15[d] : (R0 == 7 ? kpc_bm7[d] : (R0 == 3 ? kpc_bm3[d] : kpc_bm1[d]));
}

// min(a, b, c) in one instruction (FMNMX3, sm_100); the same value as fminf(fminf(a, b), c)
__device__ __forceinline__ float kp_min3(float a, float b, float c)
{
    float r;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}

// Launch constants of the score filter, converted once per kernel (every caller of kp_score_lower_bound2 takes them from
// here).  base = the margin's constant term: 0.01, plus 4e-4 |penalty| when penalty < 0.  The relative term rel |est| of
// the margin only bounds the error when est = pen + t1 + t2 does not cancel, i.e. pen >= 0; with pen < 0 the error still
// scales with t1 + t2 = est - pen <= |est| + |pen|, so rel (t1 + t2 + |pen|) <= rel |est| + 2 rel |pen| <= rel |est| +
// 4e-4 |pen| for both values of rel, which also covers the rounding of penalty to float32.
struct KpFilterK { float alpha, ab, penalty, base; };
__device__ __forceinline__ KpFilterK kp_filter_consts(double alpha, double beta, double penalty)
{
    KpFilterK f;
    f.alpha = (float)alpha;
    f.ab = (float)(alpha + beta);
    f.penalty = (float)penalty;
    f.base = penalty >= 0.0 ? 0.01f : __fmaf_rn(4e-4f, (float)-penalty, 0.01f);
    return f;
}

// Float32 lower bound of the self-score (w_numba.py:56-61) for the score filter, two patterns at a time with
// the packed f32x2 instructions of sm_100 (FADD2/FMUL2/FFMA2).  Error budget of the estimate (pen >= 0: both terms of s
// are >= 0, no cancellation; pen < 0: see kp_filter_consts):
//   counts -> float32 and their sums   <= 4 roundings of 2^-24 on M, U           (exact below 2^24)
//   p = (M + a) / (M + U + a + b)      <= 2 roundings + __fdividef (2 ulp):  |dp| / p <= 2.4e-7 + conversions 3.6e-7 = 6e-7
//   p < 2^-5 (the usual case):  ln p < -3.4, so  __logf  is in its RELATIVE regime (3 ulp) and the error of p adds
//       6e-7 / 3.4 relative: 5.5e-7 of the first term; ln(1-p) by its series (truncation p^4/5 < 2e-7, three roundings) plus the
//       error of p: 1e-6 of the second term; the final fma / mul / add: 2e-7.   Total < 1.5e-6 |s|.  Not relative: s is the
//       reference's float64 score, whose q = 1 - p is rounded by up to 2^-54, so its -2U ln q is off by up to U 2^-53 however
//       small p is (for p < 2^-54 it is 0 instead of 2Up); with counts above 2^46 that exceeds 0.01.
//       Bound used: 1e-5 |s| + 2^-52 (M + U) + 0.01.
//   p >= 2^-5:  __logf has ABSOLUTE error 2^-21.4 = 3.6e-7 for arguments in [0.5, 2] (rates near 1, or 1-p above the series
//       range), and the error of p enters ln p and ln(1-p) absolutely (up to 6e-7 / 0.5): together < 1.6e-6 per unit of count,
//       times 2: bound used  2e-4 |s| + 4e-6 (M + U) + 0.01.
// A NaN (p == 0, ...) never skips the exact score.  tests/test_gpu_score_bounds.py checks lb <= s at the edges.
__device__ __forceinline__ float2 kp_score_lower_bound2(float2 Mf, float2 Uf, const KpFilterK &f)
{
    const float2 num = __fadd2_rn(Mf, make_float2(f.alpha, f.alpha));
    const float2 cnt = __fadd2_rn(Mf, Uf);
    const float2 den = __fadd2_rn(cnt, make_float2(f.ab, f.ab));
    const float2 p = make_float2(__fdividef(num.x, den.x), __fdividef(num.y, den.y));
    const float2 lp = make_float2(__logf(p.x), __logf(p.y));
    // log(1-p) = -p (1 + p (1/2 + p (1/3 + p/4)))  for p < 2^-5
    float2 t = __ffma2_rn(p, make_float2(0.25f, 0.25f), make_float2(0.33333334f, 0.33333334f));
    t = __ffma2_rn(p, t, make_float2(0.5f, 0.5f));
    t = __ffma2_rn(p, t, make_float2(1.0f, 1.0f));
    float2 l1 = __fmul2_rn(make_float2(-p.x, -p.y), t);
    float2 rel = make_float2(1e-5f, 1e-5f), per = make_float2(0x1p-52f, 0x1p-52f);   // margin of the small rates
    if (!(p.x < 0.03125f)) { l1.x = __logf(1.0f - p.x); rel.x = 2e-4f; per.x = 4e-6f; }
    if (!(p.y < 0.03125f)) { l1.y = __logf(1.0f - p.y); rel.y = 2e-4f; per.y = 4e-6f; }
    const float2 ll = __ffma2_rn(Mf, lp, __fmul2_rn(Uf, l1));                       // M log p + U log(1-p)  (<= 0)
    const float2 est = __ffma2_rn(ll, make_float2(-2.0f, -2.0f), make_float2(f.penalty, f.penalty));
    const float2 mar = __ffma2_rn(make_float2(fabsf(est.x), fabsf(est.y)), rel, __ffma2_rn(cnt, per, make_float2(f.base, f.base)));
    return __fadd2_rn(est, make_float2(-mar.x, -mar.y));
}

// 16-byte read-only load with an L2 cache policy (createpolicy): used for child tiles nobody re-reads while they could
// still be in L2 (children along the top tile position: their other parents are thousands of tiles away in the claim
// order), so that they do not push out the lines sibling tiles are about to share
__device__ __forceinline__ float4 kp_ldg_policy(const float4 *ptr, unsigned long long policy)
{
    float4 v;
    asm("ld.global.nc.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
        : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(ptr), "l"(policy));
    return v;
}

// ---------------------------------------------------------------------------------------------------
// K3+K4: lazily fused self-score + min-plus recurrence
// ---------------------------------------------------------------------------------------------------
// Where the tiles of a score table live: one table, or one shard per GPU of the node (SURVEY 8f.3).  A table is
// sharded by the digit of the TOP high position (the most significant one of the tile number): the tiles of digit d
// belong to rank owner[d] and are stored there as if the digit were slot[d].  nshard == 1: hw_top = ntiles, so
// the digit is 0 for every tile and owner[0] = slot[0] = 0.
#define KP_MAX_SHARDS 8
struct KpView {
    const float *best[KP_MAX_SHARDS];        // (peer) pointers to every rank's shard of the score table
    const uint16_t *flags[KP_MAX_SHARDS];    // ... and of the kept-whole flags
    uint32_t hw_top;
    uint8_t owner[16], slot[16];
    uint8_t push_mask[16];   // replicated mode: ranks (bit r) that own a strict superset of the digit, i.e. read its tiles
    // replicated mode, two-dimensional ownership (general patterns with at least two high positions): the owner of a tile
    // depends on the digits of the TWO top high positions, cell = tile / hw_second = d_second + radix_second * d_top.
    // Spreads the inbound NVLink traffic, which with one-dimensional ownership piles up on the owner of digit N.
    uint32_t hw_second;
    uint32_t two_d;
    uint8_t owner2[256];     // cell -> owner rank
    uint8_t push_mask2[256]; // cell -> ranks that own a parent of the cell's tiles along either of the two positions
};

__device__ __forceinline__ void kp_view_tile(const KpView &v, unsigned long long tile, int &rank, unsigned long long &ltile)
{
    if (v.two_d) {   // replicated tables hold global tile numbers
        rank = v.owner2[tile / v.hw_second];
        ltile = tile;
        return;
    }
    const unsigned long long d = tile / v.hw_top;
    rank = v.owner[d];
    ltile = (unsigned long long)v.slot[d] * v.hw_top + (tile - d * v.hw_top);
}

struct KpDpParams {
    const KpTables *tab;
    const uint8_t *rowtab;
    const uint32_t *tile_list;  // tiles of this wave, ascending
    uint32_t ntiles_wave;
    uint32_t *counter;          // next unclaimed entry of tile_list (zeroed before the launch)
    int leaf_wave;              // wave 0: rows of level 0 hold k-mers at the single-nucleotide digits
    int pf_dist;                // L2 prefetch distance of the child-tile stream, in (32 rows x 1 split) steps
    int evict_top;              // child tiles along the top `evict_top` high positions are loaded with an L2 evict-first policy
    int pf_top;                 // only the splits of the top `pf_top` high positions are prefetched into L2 (<= 0: all of them)
    int pf_bulk;                // L2 prefetch by bulk copies (cp.async.bulk.prefetch.L2, one per 512-byte segment) instead of one line per lane
    const long long *e0, *e1;   // expanded counts M, U  [ntiles][tile_kmers]
    const long long *s0, *s1;   // CV job: held-out expanded counts, subtracted on the fly (train = total - held-out); else null
    double alpha, beta, penalty;
    float *best;                // best loss per pattern (sharded: this rank's shard)
    uint16_t *flags;            // per row, bit d set = pattern kept whole
    KpView view;                // sharded DP only: every rank's shard, for the child tiles of the top position
    int my_rank;
    // single-launch mode (SHARD == 3): all waves in one launch, a tile waits for its child tiles instead of a
    // kernel boundary, so the tail of one wave overlaps the head of the next
    const uint8_t *tile_wave;   // wave of every entry of tile_list
    uint8_t *tile_done;         // [ntiles] 1 once a tile's rows are stored (zeroed before the launch)
    uint32_t *wave_done;        // [64] finished tiles per wave (zeroed before the launch)
    uint32_t wave_size[64];     // tiles per wave
    int *err;                   // set when a dependency wait gives up (never expected)
};

// RP: the row pitch as a compile-time constant (0: read it from the tables).  With the pitch known, the tile
// stride and the four group offsets of a row fold into immediates of the child-tile loads.
// SHARD: the tiles are split over the GPUs of the node by the digit of the top high position.
//   1 (partitioned, capacity): every rank stores its own tiles only; a tile's children along the top position may
//     live in a peer's memory and are then loaded over NVLink by the same pipeline (split lists carry the owner
//     rank in their top 4 bits).
//   2 (replicated, speed): every rank holds a full-size table; a finished row is stored locally AND into the
//     table of every peer that owns a superset digit (posted NVLink writes), so all reads stay local.
//   4 (one GPU, small waves): at most one tile per SM in the wave (the last waves of a big lattice, every wave of a small one).
//     A CTA owns one tile: each of its warps streams ONE 32-row chunk of the child tiles into the shared copy, then warp 0
//     runs the rounds; the wave then costs a fraction of a tile latency instead of a whole one.
//   3 (one GPU, single launch; opt-in): tile_list holds every wave back to back and tiles are claimed in that order by
//     the resident warps (one CTA per SM, all resident); a tile spins until its child tiles are flagged done.  Claiming
//     in order makes this deadlock-free: every child was claimed earlier, by a warp that is running.  The table is then
//     written and read by the same kernel, so its loads are ld.global.cg instead of the read-only (.nc) path - which
//     costs more than the overlapped wave tails gain in a sustained run (DESIGN.md section 4).
template <int R0, bool WIDE, int RP, int SHARD>
__global__ void KP_DP_BOUNDS kp_dp_rows_kernel(const KpDpParams p)
{
    typedef typename KpCnt<WIDE>::type C;
    constexpr int NG = (R0 + 3) / 4;
    constexpr int NB = R0 == 15 ? 4 : (R0 == 7 ? 3 : (R0 == 3 ? 2 : 1));
    constexpr bool SHARDED = SHARD == 1;   // partitioned addressing
    constexpr bool ONE_LAUNCH = SHARD == 3;
    constexpr bool COOP = SHARD == 4;      // one tile per CTA: every warp streams one 32-row chunk, warp 0 runs the rounds

    extern __shared__ __align__(16) unsigned char smem[];
    const KpTables &tb = *p.tab;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rp = RP ? RP : tb.rp, nrounds = tb.nrounds, nhigh = tb.nhigh, nrows = tb.nrows;
    const uint32_t stride = RP ? (uint32_t)(NG * RP * 4) : tb.tile_stride, tk = tb.tile_kmers;
    const uint32_t rt_bytes = tb.rt_bytes;
    const int maxhs = tb.maxhs;

    double2 *logtab = (double2 *)smem;
    unsigned char *rt = smem + 2048;
    for (int i = threadIdx.x; i < 128; i += blockDim.x) logtab[i] = make_double2(kpc_logTab[2 * i], kpc_logTab[2 * i + 1]);
    for (uint32_t i = threadIdx.x; i < rt_bytes / 4; i += blockDim.x) ((uint32_t *)rt)[i] = ((const uint32_t *)p.rowtab)[i];
    __syncthreads();
    const uint16_t *round_start = (const uint16_t *)(rt + tb.rt_round_start);
    const uint8_t *row_level = rt + tb.rt_row_level;
    const uint16_t *xs_off = (const uint16_t *)(rt + tb.rt_xs_off);
    const uint32_t *xs = (const uint32_t *)(rt + tb.rt_xs);
    const uint16_t *bs_off = (const uint16_t *)(rt + tb.rt_bs_off);
    const uint16_t *bs = (const uint16_t *)(rt + tb.rt_bs);

    unsigned char *wm = smem + 2048 + rt_bytes + (size_t)(COOP ? 0 : warp) * tb.warp_smem_bytes[WIDE];
    float4 *S = (float4 *)wm;                                  // [NG][rp] the warp's copy of its tile
    C *bc = (C *)(wm + (size_t)NG * rp * 16);                  // [tile_kmers][2] base counts of the tile
    uint32_t *hs1 = (uint32_t *)((unsigned char *)bc + (size_t)tk * 2 * sizeof(C));
    uint32_t *hs2 = hs1 + maxhs;
    int *s_nhs = (int *)(hs2 + maxhs);
    const double alpha = p.alpha, beta = p.beta, penalty = p.penalty;
    const KpFilterK fk = kp_filter_consts(alpha, beta, penalty);
    const float INF = __int_as_float(0x7f800000);
    const float *tbase = p.best;
    unsigned long long pol_first;
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol_first));

    // Tiles are claimed in list order (ascending tile number): the tiles in flight on the whole GPU are then
    // always neighbours in the pattern lattice, which share child tiles, so those re-reads hit in L2.
    for (;;) {
        uint32_t it = 0;
        if (COOP) {   // the CTA claims: all warps have left the previous tile, then one thread takes the next
            __syncthreads();
            if (threadIdx.x == 0) s_nhs[3] = (int)atomicAdd(p.counter, 1u);
            __syncthreads();
            it = (uint32_t)s_nhs[3];
        } else {
            if (lane == 0) it = atomicAdd(p.counter, 1u);
            it = __shfl_sync(0xffffffffu, it, 0);
        }
        if (it >= p.ntiles_wave) break;
        const uint32_t tile = p.tile_list[it];
        const int wave = ONE_LAUNCH ? (int)p.tile_wave[it] : 0;
        const bool leaf_tile = ONE_LAUNCH ? wave == 0 : (p.leaf_wave != 0);
        uint32_t ltile = tile;   // index of the tile in this rank's table
        if (SHARDED) {
            const uint32_t dt = tile / p.view.hw_top;
            ltile = (uint32_t)p.view.slot[dt] * p.view.hw_top + (tile - dt * p.view.hw_top);
        }
        __syncwarp();  // previous tile's readers of S / bc / hs are done
        // ---- the tile's high-position splits (two child tiles each) ----
        if (!COOP || warp == 0) {
            int ns = 0, d = 0, e = 0;
            uint32_t m = 0, hw = 1;
            if (lane < nhigh) {
                e = tb.highpos[lane];
                hw = tb.highw[e];
                d = (int)((tile / hw) % tb.radix[e]);
                m = tb.digit_mask[e][d];
                ns = tb.ms_n[m];
            }
            int off = ns;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int x = __shfl_up_sync(0xffffffffu, off, o);
                if (lane >= o) off += x;
            }
            int total = __shfl_sync(0xffffffffu, off, 31);
            off -= ns;
            for (int j = 0; j < ns; j++) {
                int c1 = tb.mask_digit[e][tb.ms_c1[m][j]], c2 = tb.mask_digit[e][tb.ms_c2[m][j]];
                if (!SHARDED) {
                    hs1[off + j] = tile - (uint32_t)(d - c1) * hw;
                    hs2[off + j] = tile - (uint32_t)(d - c2) * hw;
                } else if (lane == nhigh - 1) {   // top position: d is the sharding digit, tile - d * hw the rest
                    const uint32_t rest = tile - (uint32_t)d * hw;
                    hs1[off + j] = ((uint32_t)p.view.slot[c1] * hw + rest) | ((uint32_t)p.view.owner[c1] << 28);
                    hs2[off + j] = ((uint32_t)p.view.slot[c2] * hw + rest) | ((uint32_t)p.view.owner[c2] << 28);
                } else {                          // same sharding digit: a local tile
                    hs1[off + j] = (ltile - (uint32_t)(d - c1) * hw) | ((uint32_t)p.my_rank << 28);
                    hs2[off + j] = (ltile - (uint32_t)(d - c2) * hw) | ((uint32_t)p.my_rank << 28);
                }
            }
            if (lane == 0) *s_nhs = total;
            if (KP_EXPERIMENTS && !SHARDED && !ONE_LAUNCH) {   // first split of the top `evict_top` positions (the list is in position order)
                const int first = nhigh - p.evict_top;
                const int ptop_ = p.evict_top > 0 ? __shfl_sync(0xffffffffu, off, first > 0 ? first : 0) : 0x7fffffff;
                if (lane == 0) s_nhs[1] = ptop_;
                // first split that gets an L2 prefetch: the children along the LOW high positions are mostly in L2 already
                // (sibling tiles just read them), so prefetching them only costs L2 look-ups
                const int pfirst = nhigh - p.pf_top;
                const int pfs_ = (p.pf_top > 0 && pfirst > 0) ? __shfl_sync(0xffffffffu, off, pfirst) : 0;
                if (lane == 0) s_nhs[2] = pfs_;
            }
        }
        if (ONE_LAUNCH && wave > 0) {
            // ---- wait for the child tiles.  They sit at most three waves back (a split lowers one position by at
            //      most three levels): if those waves are complete nothing needs checking ----
            bool all_done = true;
            if (lane < 3 && wave - 1 - lane >= 0) {
                const int w = wave - 1 - lane;
                uint32_t c;
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(c) : "l"(p.wave_done + w) : "memory");
                all_done = c == p.wave_size[w];
            }
            all_done = __all_sync(0xffffffffu, all_done);   // one decision for the warp
            if (!all_done) {
                __syncwarp();   // split lists written by the other lanes
                const int n2 = 2 * *s_nhs;
                for (int j = lane; j < n2; j += 32) {
                    const uint32_t child = j & 1 ? hs2[j >> 1] : hs1[j >> 1];
                    unsigned spins = 0;
                    for (;;) {
                        uint32_t f;
                        asm volatile("ld.acquire.gpu.global.u8 %0, [%1];" : "=r"(f) : "l"(p.tile_done + child) : "memory");
                        if (f) break;
                        if (++spins > (1u << 22)) { atomicExch(p.err, 2); break; }
                        __nanosleep(200);
                    }
                }
            }
        }
        // ---- base counts of the tile ----
        for (uint32_t kl = COOP ? threadIdx.x : lane; kl < tk; kl += COOP ? blockDim.x : 32) {
            size_t g = (size_t)tile * tk + kl;
            bc[kl * 2 + 0] = (C)(p.s0 ? p.e0[g] - p.s0[g] : p.e0[g]);
            bc[kl * 2 + 1] = (C)(p.s1 ? p.e1[g] - p.s1[g] : p.e1[g]);
        }
        __syncwarp();
        if (COOP) __syncthreads();   // split list (warp 0) and base counts (all warps) are in place
        const int nhs = *s_nhs;
        const int ptop = (KP_EXPERIMENTS && !SHARDED && !ONE_LAUNCH) ? s_nhs[1] : 0x7fffffff;
        const int pfs = (KP_EXPERIMENTS && !SHARDED && !ONE_LAUNCH) ? s_nhs[2] : 0;
        float4 *otile = (float4 *)(p.best + (size_t)ltile * stride);
        uint32_t pushm = 0;   // replicated mode: peers that will read this tile
        if (SHARD == 2) pushm = p.view.two_d ? p.view.push_mask2[tile / p.view.hw_second] : p.view.push_mask[tile / p.view.hw_top];

        // ---- phase D: stream the child tiles of the high-position splits for ALL rows of the tile; the running
        //      minimum of row r is parked in S[r] until the row's turn in the schedule.  One flattened software
        //      pipeline over (32-row chunk, split): a load is always two steps ahead of its use, also across
        //      chunk boundaries, so the pipeline drains once per tile ----
        {
            float v[NG * 4];
#pragma unroll
            for (int c = 0; c < NG * 4; c++) v[c] = INF;
            const int nchunk_all = (nrows + 31) >> 5;
            const int chunk0 = COOP ? warp : 0;                                   // first 32-row chunk this warp streams
            const int nchunk = COOP ? (warp < nchunk_all ? 1 : 0) : nchunk_all;   // ... and how many
            const int pend = COOP ? (nrows < 32 * (chunk0 + 1) ? nrows : 32 * (chunk0 + 1)) : nrows;   // end of its rows
            const int nstep = nhs > 0 ? nchunk * nhs : 0;
            float4 xa0[NG], xb0[NG], xa1[NG], xb1[NG];
#if KP_PIPE_DEPTH == 3
            float4 xa2[NG], xb2[NG];
#endif
            const float4 *tb4 = (const float4 *)tbase;
            const uint32_t stride4 = stride >> 2;                 // tile stride in float4
            int ls = 0, lrow = lane + 32 * chunk0;          // split and row of the next load
            const float4 *lptr = tb4 + (lrow < nrows ? lrow : nrows - 1);   // idle lanes of the last chunk re-read a valid row
            int lrowc = lrow < nrows ? lrow : nrows - 1;                    // (sharded: the row, the base depends on the owner)
            int us = 0, urow = lane + 32 * chunk0;          // split and row of the next use
            // register-free deepening of the pipeline: every step also asks L2 for the lines of a later step.
            // One prefetch per step: the 2 x NG x 4 lines (128 B = 8 rows) of a step map onto the 32 lanes.
            int ps = 0, pchunk = 32 * chunk0;   // split and first row of the next L2 prefetch (pf_dist steps ahead)
            const uint32_t *pf_hs = (lane & 16) ? hs2 : hs1;
            const int pf_g = (lane >> 2) & 3, pf_line = (lane & 3) * 8;
            const float4 *pf_ptr = tb4 + pf_g * rp + pf_line;
            const bool pf_bulk = KP_EXPERIMENTS && p.pf_bulk != 0;
            const bool pf_on = (pf_bulk || pf_g < NG) && p.pf_dist >= 0;   // KP_PF_DIST < 0: no L2 prefetch at all
#define KP_FL_PREFETCH()                                                                              \
    if (pchunk < pend) {                                                                              \
        if (KP_EXPERIMENTS && !SHARDED && pf_bulk) {   /* one bulk L2 prefetch (UBLKPF) per 512-byte segment: warp-uniform addresses */ \
            if (pf_on && ps >= pfs) {                                                                 \
                const uint32_t nb_ = (uint32_t)(nrows - pchunk < 32 ? nrows - pchunk : 32) * 16u;     \
                const float4 *c1_ = tb4 + (size_t)hs1[ps] * stride4 + pchunk, *c2_ = tb4 + (size_t)hs2[ps] * stride4 + pchunk; \
                _Pragma("unroll") for (int g = 0; g < NG; g++) {                                      \
                    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(c1_ + g * rp), "r"(nb_)); \
                    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(c2_ + g * rp), "r"(nb_)); \
                }                                                                                     \
            }                                                                                         \
        } else {                                                                                      \
            const uint32_t ph_ = pf_hs[ps];                                                           \
            if (pf_on && ps >= pfs && pchunk + pf_line < nrows && (!SHARDED || (int)(ph_ >> 28) == p.my_rank)) \
                asm volatile("prefetch.global.L2 [%0];" ::"l"(pf_ptr + (size_t)(SHARDED ? (ph_ & 0x0fffffffu) : ph_) * stride4 + pchunk)); \
        }                                                                                             \
        if (++ps == nhs) { ps = 0; pchunk += 32; }                                                    \
    }
#define KP_FL_LOAD(xa, xb)                                                                            \
    {                                                                                                 \
        KP_FL_PREFETCH()                                                                              \
        const float4 *a_, *b_;                                                                        \
        if (!SHARDED) {                                                                               \
            a_ = lptr + (size_t)hs1[ls] * stride4;                                                    \
            b_ = lptr + (size_t)hs2[ls] * stride4;                                                    \
        } else {   /* the child tile may live in a peer's memory: same load, NVLink instead of HBM */  \
            const uint32_t h1_ = hs1[ls], h2_ = hs2[ls];                                              \
            a_ = (const float4 *)p.view.best[h1_ >> 28] + lrowc + (size_t)(h1_ & 0x0fffffffu) * stride4; \
            b_ = (const float4 *)p.view.best[h2_ >> 28] + lrowc + (size_t)(h2_ & 0x0fffffffu) * stride4; \
        }                                                                                             \
        if (KP_EXPERIMENTS && !SHARDED && !ONE_LAUNCH && ls >= ptop) {   /* warp-uniform: no sibling will find these lines in L2 */ \
            _Pragma("unroll") for (int g = 0; g < NG; g++) {                                          \
                xa[g] = kp_ldg_policy(a_ + g * rp, pol_first);                                        \
                xb[g] = kp_ldg_policy(b_ + g * rp, pol_first);                                        \
            }                                                                                         \
        } else {                                                                                      \
            _Pragma("unroll") for (int g = 0; g < NG; g++) {   /* single launch: the table is written by this kernel, no .nc */ \
                xa[g] = ONE_LAUNCH ? __ldcg(a_ + g * rp) : __ldg(a_ + g * rp);                        \
                xb[g] = ONE_LAUNCH ? __ldcg(b_ + g * rp) : __ldg(b_ + g * rp);                        \
            }                                                                                         \
        }                                                                                             \
        if (++ls == nhs) {                                                                            \
            ls = 0; lrow += 32;                                                                       \
            lrowc = lrow < nrows ? lrow : nrows - 1;                                                  \
            lptr = tb4 + lrowc;                                                                       \
        }                                                                                             \
    }
#define KP_FL_USE(xa, xb)                                                                             \
    {                                                                                                 \
        _Pragma("unroll") for (int g = 0; g < NG; g++) {   /* packed f32x2 adds (FADD2), IEEE round-to-nearest */ \
            const float2 lo_ = __fadd2_rn(make_float2(xa[g].x, xa[g].y), make_float2(xb[g].x, xb[g].y)); \
            const float2 hi_ = __fadd2_rn(make_float2(xa[g].z, xa[g].w), make_float2(xb[g].z, xb[g].w)); \
            v[4 * g + 0] = fminf(v[4 * g + 0], lo_.x);                                                \
            v[4 * g + 1] = fminf(v[4 * g + 1], lo_.y);                                                \
            v[4 * g + 2] = fminf(v[4 * g + 2], hi_.x);                                                \
            v[4 * g + 3] = fminf(v[4 * g + 3], hi_.y);                                                \
        }                                                                                             \
        if (++us == nhs) {   /* chunk complete: park its minima, start the next chunk */              \
            if (urow < nrows) {                                                                       \
                _Pragma("unroll") for (int g = 0; g < NG; g++)                                        \
                    S[g * rp + urow] = make_float4(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]); \
            }                                                                                         \
            _Pragma("unroll") for (int c = 0; c < NG * 4; c++) v[c] = INF;                            \
            us = 0; urow += 32;                                                                       \
        }                                                                                             \
    }
#if KP_PIPE_DEPTH == 3
            if (nstep > 0) {
                for (int i = 0; i < p.pf_dist; i++) KP_FL_PREFETCH()
                KP_FL_LOAD(xa0, xb0)
                if (nstep > 1) KP_FL_LOAD(xa1, xb1)
            }
            for (int t = 0; t < nstep; t += 3) {   // a load is always two steps ahead of its use
                if (t + 2 < nstep) KP_FL_LOAD(xa2, xb2)
                KP_FL_USE(xa0, xb0)
                if (t + 3 < nstep) KP_FL_LOAD(xa0, xb0)
                if (t + 1 < nstep) KP_FL_USE(xa1, xb1)
                if (t + 4 < nstep) KP_FL_LOAD(xa1, xb1)
                if (t + 2 < nstep) KP_FL_USE(xa2, xb2)
            }
#else
            if (nstep > 0) {
                for (int i = 0; i < p.pf_dist; i++) KP_FL_PREFETCH()
                KP_FL_LOAD(xa0, xb0)
            }
            int t = 0;
            for (; t + 2 <= nstep; t += 2) {
                KP_FL_LOAD(xa1, xb1)
                KP_FL_USE(xa0, xb0)
                if (t + 2 < nstep) KP_FL_LOAD(xa0, xb0)
                KP_FL_USE(xa1, xb1)
            }
            if (t < nstep) KP_FL_USE(xa0, xb0)
#endif
#undef KP_FL_LOAD
#undef KP_FL_USE
#undef KP_FL_PREFETCH
            if (nhs <= 0)  // no high-position split (wave 0, or a pattern without high positions)
                for (int srow = COOP ? (int)threadIdx.x : lane; srow < nrows; srow += COOP ? (int)blockDim.x : 32) {
#pragma unroll
                    for (int g = 0; g < NG; g++) S[g * rp + srow] = make_float4(INF, INF, INF, INF);
                }
            __syncwarp();
            if (COOP) __syncthreads();   // every chunk's minima are parked
        }

        // ---- rounds ----
        for (int rnd = 0; rnd < (COOP && warp != 0 ? 0 : nrounds); rnd++) {
            const int srow = round_start[rnd] + lane;
            if (srow < round_start[rnd + 1]) {
                float v[NG * 4];
#pragma unroll
                for (int g = 0; g < NG; g++) {  // minimum over the high-position splits, parked by phase D
                    float4 x = S[g * rp + srow];
                    v[4 * g] = x.x; v[4 * g + 1] = x.y; v[4 * g + 2] = x.z; v[4 * g + 3] = x.w;
                }
                // ---- cross-row splits: finished rows of this tile, shared memory ----
                {
                    int i = xs_off[srow];
                    const int iend = xs_off[srow + 1];
                    for (; i + 2 <= iend; i += 2) {   // two splits per pass: one 3-input min per cell
                        const uint32_t pr = xs[i], pq = xs[i + 1];
                        const float4 *a = S + (pr & 0xFFFFu), *b = S + (pr >> 16);
                        const float4 *c = S + (pq & 0xFFFFu), *e = S + (pq >> 16);
#pragma unroll
                        for (int g = 0; g < NG; g++) {
                            const float4 xa = a[g * rp], xb = b[g * rp], xc = c[g * rp], xe = e[g * rp];
                            const float2 l1 = __fadd2_rn(make_float2(xa.x, xa.y), make_float2(xb.x, xb.y));
                            const float2 h1 = __fadd2_rn(make_float2(xa.z, xa.w), make_float2(xb.z, xb.w));
                            const float2 l2 = __fadd2_rn(make_float2(xc.x, xc.y), make_float2(xe.x, xe.y));
                            const float2 h2 = __fadd2_rn(make_float2(xc.z, xc.w), make_float2(xe.z, xe.w));
                            v[4 * g + 0] = kp_min3(v[4 * g + 0], l1.x, l2.x);
                            v[4 * g + 1] = kp_min3(v[4 * g + 1], l1.y, l2.y);
                            v[4 * g + 2] = kp_min3(v[4 * g + 2], h1.x, h2.x);
                            v[4 * g + 3] = kp_min3(v[4 * g + 3], h1.y, h2.y);
                        }
                    }
                    if (i < iend) {
                        const uint32_t pr = xs[i];
                        const float4 *a = S + (pr & 0xFFFFu), *b = S + (pr >> 16);
#pragma unroll
                        for (int g = 0; g < NG; g++) {
                            const float4 xa = a[g * rp], xb = b[g * rp];
                            const float2 lo_ = __fadd2_rn(make_float2(xa.x, xa.y), make_float2(xb.x, xb.y));
                            const float2 hi_ = __fadd2_rn(make_float2(xa.z, xa.w), make_float2(xb.z, xb.w));
                            v[4 * g + 0] = fminf(v[4 * g + 0], lo_.x);
                            v[4 * g + 1] = fminf(v[4 * g + 1], lo_.y);
                            v[4 * g + 2] = fminf(v[4 * g + 2], hi_.x);
                            v[4 * g + 3] = fminf(v[4 * g + 3], hi_.y);
                        }
                    }
                }
                // ---- counts of this row at the single-nucleotide digits of the register position ----
                C m[NB], u[NB];
#pragma unroll
                for (int b = 0; b < NB; b++) { m[b] = 0; u[b] = 0; }
                for (int i = bs_off[srow]; i < bs_off[srow + 1]; i++) {
                    const C *q = bc + (size_t)bs[i] * NB * 2;   // {M, U} of the NB k-mers of a base row: NB * 2 * sizeof(C) bytes
                    if (!WIDE && NB % 2 == 0) {                 // 16-byte aligned: two k-mers per load
#pragma unroll
                        for (int b = 0; b < NB; b += 2) {
                            const uint4 x = *(const uint4 *)(q + b * 2);
                            m[b] += x.x; u[b] += x.y; m[b + 1] += x.z; u[b + 1] += x.w;
                        }
                    } else {
#pragma unroll
                        for (int b = 0; b < NB; b++) { m[b] += q[b * 2 + 0]; u[b] += q[b * 2 + 1]; }
                    }
                }
                // ---- score filter: which patterns can still be kept whole? (v only decreases from here) ----
                const bool leafrow = leaf_tile && row_level[srow] == 0;
                uint32_t need = 0;
                {
                    float mf[NB], uf[NB];
#pragma unroll
                    for (int b = 0; b < NB; b++) { mf[b] = (float)m[b]; uf[b] = (float)u[b]; }
#pragma unroll
                    for (int h = 0; h < (R0 + 1) / 2; h++) {   // two digits per evaluation
                        float2 Mf = make_float2(0.f, 0.f), Uf = make_float2(0.f, 0.f);
#pragma unroll
                        for (int b = 0; b < NB; b++) {
                            if ((kp_bm_c<R0>(2 * h) >> b) & 1) { Mf.x += mf[b]; Uf.x += uf[b]; }
                            if (2 * h + 1 < R0 && ((kp_bm_c<R0>(2 * h + 1) >> b) & 1)) { Mf.y += mf[b]; Uf.y += uf[b]; }
                        }
                        const float2 lb = kp_score_lower_bound2(Mf, Uf, fk);
                        if (!(lb.x > v[2 * h])) need |= 1u << (2 * h);
                        if (2 * h + 1 < R0 && !(lb.y > v[2 * h + 1])) need |= 1u << (2 * h + 1);
                    }
                    if (leafrow) need |= (1u << NB) - 1u;
                }
                // ---- exact float64 self-score of the patterns that passed the filter ----
                float sfx[NG * 4];   // one register per digit: written below by compile-time index under a predicate
#pragma unroll
                for (int c = 0; c < NG * 4; c++) sfx[c] = 0.f;
                uint32_t rupm = 0;
                if (need) {
                    const KpLogK K = kp_logk_load();
                    uint32_t todo = need;
                    while (todo) {
                        const int d = __ffs(todo) - 1;
                        todo &= todo - 1;
                        const unsigned bm = kp_bm<R0>(d);
                        C M_ = 0, U_ = 0;
#pragma unroll
                        for (int b = 0; b < NB; b++)
                            if ((bm >> b) & 1u) { M_ += m[b]; U_ += u[b]; }
                        float sf;
                        bool ru;
                        const bool leafcell = leafrow && d < NB;
                        if (leafcell || !kp_self_score_fast<C>(M_, U_, alpha, beta, penalty, logtab, K, sf, ru)) {
                            // k-mers (scipy's formula), and the one score in 10^5 the fast bound cannot decide: exact
                            const double s_ = leafcell ? kp_leaf_score_nl(M_, U_, alpha, beta, penalty, logtab)
                                                       : kp_self_score_exact_nl<C>(M_, U_, alpha, beta, penalty, logtab);
                            sf = __double2float_rn(s_);
                            ru = (double)sf > s_;
                        }
                        if (ru) rupm |= 1u << d;
                        // park the result in this row's own slot of S (its minima are in v[] since the start of the round and
                        // the slot is rewritten by the row's final store): one 4-byte store instead of R0 predicated moves
                        ((float *)(S + (d >> 2) * rp + srow))[d & 3] = sf;
                    }
#pragma unroll
                    for (int g = 0; g < NG; g++) {
                        const float4 x = S[g * rp + srow];
                        sfx[4 * g] = x.x; sfx[4 * g + 1] = x.y; sfx[4 * g + 2] = x.z; sfx[4 * g + 3] = x.w;
                    }
                }
                // ---- register position: in-register splits + self-score compare, digit by digit.
                //      reference: if s < (double)best: best = f32(s)   <=>   sf < best || (sf == best && sf > s) ----
                uint32_t flag = 0;
#define KP_FIN(D)                                                                                     \
    if ((need >> (D)) & 1u) {                                                                         \
        const float sf_ = sfx[D];                                                                     \
        if (sf_ < v[D] || (sf_ == v[D] && ((rupm >> (D)) & 1u))) { v[D] = sf_; flag |= 1u << (D); }   \
    }
#define KP_SP(D, A, B) v[D] = fminf(v[D], __fadd_rn(v[A], v[B]));
#define KP_SP2(D, A, B, A2, B2) v[D] = kp_min3(v[D], __fadd_rn(v[A], v[B]), __fadd_rn(v[A2], v[B2]));
                if (R0 == 1) {
                    KP_FIN(0)
                } else if (R0 == 3) {
                    KP_FIN(0) KP_FIN(1)
                    KP_SP(2, 0, 1) KP_FIN(2)
                } else if (R0 == 7) {
                    KP_FIN(0) KP_FIN(1) KP_FIN(2)
                    KP_SP(3, 0, 1) KP_FIN(3)
                    KP_SP(4, 0, 2) KP_FIN(4)
                    KP_SP(5, 1, 2) KP_FIN(5)
                    KP_SP2(6, 0, 5, 1, 4) KP_SP(6, 2, 3) KP_FIN(6)
                } else {
                    KP_FIN(0) KP_FIN(1) KP_FIN(2) KP_FIN(3)
                    KP_SP(4, 0, 2) KP_FIN(4)     // R = A|G
                    KP_SP(5, 1, 3) KP_FIN(5)     // Y = C|T
                    KP_SP(6, 2, 1) KP_FIN(6)     // S = G|C
                    KP_SP(7, 0, 3) KP_FIN(7)     // W = A|T
                    KP_SP(8, 2, 3) KP_FIN(8)     // K = G|T
                    KP_SP(9, 0, 1) KP_FIN(9)     // M = A|C
                    KP_SP2(10, 1, 8, 2, 5) KP_SP(10, 3, 6) KP_FIN(10)   // B
                    KP_SP2(11, 0, 8, 2, 7) KP_SP(11, 3, 4) KP_FIN(11)   // D
                    KP_SP2(12, 0, 5, 1, 7) KP_SP(12, 3, 9) KP_FIN(12)   // H
                    KP_SP2(13, 0, 6, 1, 4) KP_SP(13, 2, 9) KP_FIN(13)   // V
                    KP_SP2(14, 6, 7, 8, 9) KP_SP2(14, 4, 5, 0, 10)
                    KP_SP2(14, 1, 11, 2, 12) KP_SP(14, 3, 13) KP_FIN(14)  // N
                }
#undef KP_FIN
#undef KP_SP
#undef KP_SP2
                // ---- store the row ----
#pragma unroll
                for (int c = R0; c < NG * 4; c++) v[c] = 0.f;
#pragma unroll
                for (int g = 0; g < NG; g++) {
                    float4 o = make_float4(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
                    S[g * rp + srow] = o;
                    __stcs(otile + g * rp + srow, o);  // next read is a whole wave away: do not keep it in L2
                }
                p.flags[(size_t)ltile * rp + srow] = (uint16_t)flag;
                if (SHARD == 2) {
                    for (uint32_t pm = pushm; pm; pm &= pm - 1) {   // posted writes into the peers' replicas
                        const int r = __ffs(pm) - 1;
                        float4 *rt_ = (float4 *)(const_cast<float *>(p.view.best[r]) + (size_t)tile * stride);
#pragma unroll
                        for (int g = 0; g < NG; g++)
                            rt_[g * rp + srow] = make_float4(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
                        const_cast<uint16_t *>(p.view.flags[r])[(size_t)tile * rp + srow] = (uint16_t)flag;
                    }
                }
            }
            __syncwarp();  // rows of this round visible to the warp
        }
        if (ONE_LAUNCH) {   // publish the tile: every lane's stores, then the flag and the wave counter
            __threadfence();
            __syncwarp();
            if (lane == 0) {
                asm volatile("st.release.gpu.global.u8 [%0], %1;" ::"l"(p.tile_done + tile), "r"(1u) : "memory");
                atomicAdd(p.wave_done + wave, 1u);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// CV job helpers.  A CV job is the DP above on the TRAIN counts (total - held-out); the held-out loss of
// the optimal partition is then summed along the partition tree (_CV.py:46-51, :71-78): a leaf contributes
// the float32 held-out loss of the unsplit pattern, an inner node the float32 sum of its two children.
// ---------------------------------------------------------------------------------------------------
// ---------------------------------------------------------------------------------------------------
// K1: scatter packed k-mers into the dense k-mer tables (duplicates add, like read_dict)
// ---------------------------------------------------------------------------------------------------
__global__ void kp_pack_kernel(const KpTables *tab, const uint8_t *gen_mask, int k, const unsigned long long *codes,
                               const long long *pos, const long long *neg, unsigned long long n, long long *kmerM,
                               long long *kmerU, int *err)
{
    const KpTables &tb = *tab;
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        unsigned long long code = codes[i];
        unsigned long long kidx = 0;
        int e = 0;
        bool ok = true;
        for (int s = 0; s < k; s++) {
            unsigned m = (unsigned)((code >> (4 * s)) & 15u);
            unsigned g = gen_mask[s];
            if (m == 0 || (m & (m - 1)) || !(m & g)) { ok = false; break; }
            if (g & (g - 1)) {  // multi-letter position: carries a digit
                kidx += (unsigned long long)tb.mask_digit[e][m] * tb.kw[e];
                e++;
            }
        }
        if (!ok || (k < 16 && (code >> (4 * k)) != 0)) { atomicExch(err, 1); continue; }
        atomicAdd((unsigned long long *)&kmerM[kidx], (unsigned long long)pos[i]);
        atomicAdd((unsigned long long *)&kmerU[kidx], (unsigned long long)neg[i]);
    }
}

// ---------------------------------------------------------------------------------------------------
// K2: expanded counts E[tile][low k-mer] = sum over the high k-mers covered by the tile's high digits
// ---------------------------------------------------------------------------------------------------
__global__ void kp_expand_base_kernel(const KpTables *tab, unsigned long long nkmer, const long long *kmerM,
                                      const long long *kmerU, long long *expM, long long *expU)
{
    const KpTables &tb = *tab;
    const uint32_t tk = tb.tile_kmers;
    for (unsigned long long x = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; x < nkmer;
         x += (unsigned long long)gridDim.x * blockDim.x) {
        unsigned long long rest = x, tile = 0, kl = 0;
        for (int e = 0; e < tb.npos; e++) {
            unsigned long long b = rest % tb.nbase[e];
            rest /= tb.nbase[e];
            if (tb.is_low[e]) kl += b * tb.lkw[e];
            else tile += b * tb.highw[e];  // single-nucleotide digit == base index
        }
        expM[tile * tk + kl] = kmerM[x];
        expU[tile * tk + kl] = kmerU[x];
    }
}

// pass over the hi-th high position: tiles whose digit there is multi-letter, whose earlier high digits are anything
// (already expanded) and whose later high digits are single nucleotides.  Only those `total` elements are enumerated.
__global__ void kp_expand_pass_kernel(const KpTables *tab, int hi, unsigned long long total, long long *expM, long long *expU)
{
    const KpTables &tb = *tab;
    // per-pass constants of the mixed-radix decode, once per CTA (the table struct lives in global memory)
    __shared__ uint32_t s_n[KP_MAXPOS], s_w[KP_MAXPOS], s_add[KP_MAXPOS];
    __shared__ uint32_t s_src[16][4];   // digit of the pass position -> tile offsets of its single-nucleotide sources
    __shared__ uint32_t s_nsrc[16];
    const int nhigh = tb.nhigh;
    const int e = tb.highpos[hi];
    const uint32_t tk = tb.tile_kmers;
    if (threadIdx.x < nhigh) {
        const int h = threadIdx.x, f = tb.highpos[h];
        const uint32_t nb = tb.nbase[f];
        s_n[h] = h < hi ? tb.radix[f] : (h == hi ? tb.radix[f] - nb : nb);
        s_add[h] = h == hi ? nb : 0;   // the pass position enumerates its multi-letter digits only
        s_w[h] = tb.highw[f];
    }
    if (threadIdx.x < 16) {
        const int d = threadIdx.x;
        int n = 0;
        if (d < tb.radix[e]) {
            const uint32_t m = tb.digit_mask[e][d];
            for (int b = 0; b < 4; b++)
                if ((m >> b) & 1u) s_src[d][n++] = (uint32_t)(d - tb.mask_digit[e][1u << b]) * tb.highw[e];
        }
        s_nsrc[d] = (uint32_t)n;
    }
    __syncthreads();
    for (unsigned long long x = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; x < total;
         x += (unsigned long long)gridDim.x * blockDim.x) {
        uint32_t kl, tile = 0, d = 0;
        if (total <= 0xFFFFFFFFull) {   // 32-bit index arithmetic (every realistic size)
            const uint32_t x32 = (uint32_t)x;
            kl = x32 % tk;
            uint32_t r = x32 / tk;
            for (int h = 0; h < nhigh; h++) {
                const uint32_t n = s_n[h];
                const uint32_t dig = r % n + s_add[h];   // a single-nucleotide digit is its base index
                r /= n;
                if (h == hi) d = dig;
                tile += dig * s_w[h];
            }
        } else {
            kl = (uint32_t)(x % tk);
            unsigned long long r = x / tk;
            for (int h = 0; h < nhigh; h++) {
                const uint32_t n = s_n[h];
                const uint32_t dig = (uint32_t)(r % n) + s_add[h];
                r /= n;
                if (h == hi) d = dig;
                tile += dig * s_w[h];
            }
        }
        long long am = 0, au = 0;
        const uint32_t ns = s_nsrc[d];
        for (uint32_t i = 0; i < ns; i++) {
            const size_t src = (size_t)(tile - s_src[d][i]) * tk + kl;
            am += expM[src];
            au += expU[src];
        }
        const size_t dst = (size_t)tile * tk + kl;
        expM[dst] = am;
        expU[dst] = au;
    }
}

// ---------------------------------------------------------------------------------------------------
// Locating a dense pattern number in the device layout, and re-deriving its split decision
// ---------------------------------------------------------------------------------------------------
struct KpLoc { unsigned long long tile; uint32_t srow, d0; };

__device__ __forceinline__ KpLoc kp_locate_dev(const KpTables &tb, const uint16_t *srow_of_row, unsigned long long pat)
{
    KpLoc L;
    L.tile = 0; L.d0 = 0;
    uint32_t row = 0;
    for (int e = 0; e < tb.npos; e++) {
        uint32_t dig = (uint32_t)((pat / tb.extw[e]) % tb.radix[e]);
        if (e == tb.estar) L.d0 = dig;
        else if (tb.is_low[e]) row += dig * tb.roww[e];
        else L.tile += (unsigned long long)dig * tb.highw[e];
    }
    L.srow = srow_of_row[row];
    return L;
}

// score / kept-whole flag of a located pattern, through the view (any shard)
__device__ __forceinline__ float kp_view_best(const KpTables &tb, const KpView &vw, unsigned long long tile, uint32_t srow, uint32_t d0)
{
    int r;
    unsigned long long lt;
    kp_view_tile(vw, tile, r, lt);
    return vw.best[r][lt * tb.tile_stride + ((size_t)(d0 >> 2) * tb.rp + srow) * 4 + (d0 & 3)];
}

__device__ __forceinline__ bool kp_view_kept(const KpTables &tb, const KpView &vw, unsigned long long tile, uint32_t srow, uint32_t d0)
{
    int r;
    unsigned long long lt;
    kp_view_tile(vw, tile, r, lt);
    return (vw.flags[r][lt * tb.rp + srow] >> d0) & 1u;
}

__device__ __forceinline__ float kp_best_at(const KpTables &tb, const uint16_t *srow_of_row, const KpView &vw,
                                            unsigned long long pat)
{
    KpLoc L = kp_locate_dev(tb, srow_of_row, pat);
    return kp_view_best(tb, vw, L.tile, L.srow, L.d0);
}

// counts of one pattern from an expanded table: sum over the base rows of its row and the bases of its digit
__device__ __forceinline__ void kp_counts_from_expanded(const KpTables &tb, const uint8_t *rowtab, const long long *eM,
                                                        const long long *eU, unsigned long long tile, uint32_t srow,
                                                        uint32_t d0, unsigned long long &M, unsigned long long &U)
{
    const uint16_t *bs_off = (const uint16_t *)(rowtab + tb.rt_bs_off);
    const uint16_t *bs = (const uint16_t *)(rowtab + tb.rt_bs);
    const uint32_t nb = (uint32_t)tb.nb0;
    const unsigned bm = tb.r0 == 15 ? kpc_bm15[d0] : (tb.r0 == 7 ? kpc_bm7[d0] : (tb.r0 == 3 ? kpc_bm3[d0] : kpc_bm1[d0]));
    M = 0; U = 0;
    for (int i = bs_off[srow]; i < bs_off[srow + 1]; i++)
        for (uint32_t b = 0; b < nb; b++)
            if ((bm >> b) & 1u) {
                size_t g = (size_t)tile * tb.tile_kmers + (size_t)bs[i] * nb + b;
                M += (unsigned long long)eM[g];
                U += (unsigned long long)eU[g];
            }
}

// held-out loss of every leaf of a backtracked partition: RN_f32 of _CV.py:73-78 (level >= 1) or :15-20 (k-mers)
__global__ void kp_cv_leaf_kernel(const KpTables *tab, const uint8_t *rowtab, const long long *eMtot, const long long *eUtot,
                                  const long long *eMte, const long long *eUte, double alpha, double beta, double penalty,
                                  const unsigned long long *pats, const unsigned long long *counts, unsigned long long cap,
                                  float *out)
{
    const KpTables &tb = *tab;
    const uint16_t *srow_of_row = (const uint16_t *)(rowtab + tb.rt_srow_of_row);
    const uint8_t *row_level = rowtab + tb.rt_row_level;
    __shared__ double2 logtab[128];
    for (int i = threadIdx.x; i < 128; i += blockDim.x) logtab[i] = make_double2(kpc_logTab[2 * i], kpc_logTab[2 * i + 1]);
    __syncthreads();
    unsigned long long n = counts[0] < cap ? counts[0] : cap;
    const KpLogK K = kp_logk_load();
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        KpLoc L = kp_locate_dev(tb, srow_of_row, pats[i]);
        unsigned long long Mtr, Utr, Mte, Ute;
        kp_counts_from_expanded(tb, rowtab, eMtot, eUtot, L.tile, L.srow, L.d0, Mtr, Utr);
        kp_counts_from_expanded(tb, rowtab, eMte, eUte, L.tile, L.srow, L.d0, Mte, Ute);
        Mtr -= Mte;   // train = total - held-out
        Utr -= Ute;
        bool kmer = row_level[L.srow] == 0 && L.d0 < (uint32_t)tb.nb0;
        unsigned long long x = L.tile;
        for (int h = 0; h < tb.nhigh; h++) {
            int e = tb.highpos[h];
            if (x % tb.radix[e] >= tb.nbase[e]) kmer = false;
            x /= tb.radix[e];
        }
        double t;
        if (kmer) {
            double s;
            kp_leaf_cv(Mtr, Utr, Mte, Ute, alpha, beta, penalty, logtab, s, t);
        } else {
            double lp, l1;
            kp_self_score_t<unsigned long long>(Mtr, Utr, alpha, beta, penalty, logtab, K, lp, l1);
            t = kp_test_ll_t<unsigned long long>(Mte, Ute, lp, l1);
        }
        out[i] = __double2float_rn(t);
    }
}

// The split the reference would have recorded for `pat` (w_numba.py:36-49, :62-64): 0xFF if the pattern is
// kept whole, else position*8 + j of the first split in scan order whose float32 child sum is the minimum.
__device__ uint8_t kp_split_code_dev(const KpTables &tb, const uint16_t *srow_of_row, const KpView &vw,
                                     unsigned long long pat, unsigned long long *c1_out, unsigned long long *c2_out)
{
    KpLoc L = kp_locate_dev(tb, srow_of_row, pat);
    if (kp_view_kept(tb, vw, L.tile, L.srow, L.d0)) return 0xFF;
    float bv = __int_as_float(0x7f800000);
    uint8_t code = 0xFF;
    for (int e = 0; e < tb.npos; e++) {
        unsigned long long w = tb.extw[e];
        int d = (int)((pat / w) % tb.radix[e]);
        uint32_t m = tb.digit_mask[e][d];
        for (int j = 0; j < tb.ms_n[m]; j++) {
            int c1 = tb.mask_digit[e][tb.ms_c1[m][j]], c2 = tb.mask_digit[e][tb.ms_c2[m][j]];
            unsigned long long p1 = pat - (unsigned long long)(d - c1) * w, p2 = pat - (unsigned long long)(d - c2) * w;
            float v = __fadd_rn(kp_best_at(tb, srow_of_row, vw, p1), kp_best_at(tb, srow_of_row, vw, p2));
            if (v < bv) { bv = v; code = (uint8_t)(tb.pos_id[e] * 8 + j); *c1_out = p1; *c2_out = p2; }
        }
    }
    return code;
}

// ---------------------------------------------------------------------------------------------------
// K5: backtrack.  Breadth-first expansion from the general pattern; each leaf carries its path key
// (0 = c1 side, 1 = c2 side, most significant bit first), so sorting by key restores the reference's
// depth-first, c1-first emission order.
// ---------------------------------------------------------------------------------------------------
struct KpBtNode { unsigned long long pat, key; };

// One launch per depth of the partition tree, one warp per node: lane e evaluates the splits of effective
// position e (their 2 x nsplit child reads are independent and overlap), then the warp takes the
// lexicographic minimum of (child sum, scan rank).  ctr: [0] leaves, [1] overflow flag, [2 + d] nodes at depth d.
__device__ __forceinline__ void kp_backtrack_level(const KpTables &tb, const uint8_t *rowtab, const KpView &vw, int depth,
                                                   const KpBtNode *cur, KpBtNode *nxt, KpBtNode *leaves,
                                                   unsigned long long cap, unsigned long long *ctr, unsigned long long ncur)
{
    const uint16_t *srow_of_row = (const uint16_t *)(rowtab + tb.rt_srow_of_row);
    const int lane = threadIdx.x & 31;
    const unsigned long long nw = (unsigned long long)gridDim.x * (blockDim.x >> 5);
    for (unsigned long long i = (unsigned long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < ncur; i += nw) {
        KpBtNode nd;   // written by another CTA one level earlier: read at L2
        nd.pat = __ldcg(&cur[i].pat);
        nd.key = __ldcg(&cur[i].key);
        // location of the node; its children differ in one digit, so they are located by a delta (no divisions)
        unsigned long long ntile = 0;
        uint32_t nrow = 0, nd0 = 0;
        for (int e = 0; e < tb.npos; e++) {
            uint32_t dig = (uint32_t)((nd.pat / tb.extw[e]) % tb.radix[e]);
            if (e == tb.estar) nd0 = dig;
            else if (tb.is_low[e]) nrow += dig * tb.roww[e];
            else ntile += (unsigned long long)dig * tb.highw[e];
        }
        KpLoc L;
        L.tile = ntile; L.d0 = nd0; L.srow = srow_of_row[nrow];
        bool kept = kp_view_kept(tb, vw, L.tile, L.srow, L.d0);
        auto child_best = [&](int e, int d, int c) -> float {
            unsigned long long ct = ntile;
            uint32_t cr = nrow, cd = nd0;
            if (e == tb.estar) cd = (uint32_t)c;
            else if (tb.is_low[e]) cr -= (uint32_t)(d - c) * tb.roww[e];
            else ct -= (unsigned long long)(d - c) * tb.highw[e];
            return kp_view_best(tb, vw, ct, srow_of_row[cr], cd);
        };
        float bv = __int_as_float(0x7f800000);
        int code = 0x7fffffff;
        unsigned long long b1 = 0, b2 = 0;
        if (!kept && lane < tb.npos) {
            const int e = lane;
            unsigned long long w = tb.extw[e];
            int d = (int)((nd.pat / w) % tb.radix[e]);
            uint32_t m = tb.digit_mask[e][d];
            const int ns = tb.ms_n[m];
            float v[7];
#pragma unroll
            for (int j = 0; j < 7; j++) {
                v[j] = __int_as_float(0x7f800000);
                if (j < ns) {
                    int c1 = tb.mask_digit[e][tb.ms_c1[m][j]], c2 = tb.mask_digit[e][tb.ms_c2[m][j]];
                    v[j] = __fadd_rn(child_best(e, d, c1), child_best(e, d, c2));
                }
            }
#pragma unroll
            for (int j = 0; j < 7; j++)
                if (j < ns && v[j] < bv) {
                    bv = v[j];
                    code = tb.pos_id[e] * 8 + j;
                    b1 = nd.pat - (unsigned long long)(d - (int)tb.mask_digit[e][tb.ms_c1[m][j]]) * w;
                    b2 = nd.pat - (unsigned long long)(d - (int)tb.mask_digit[e][tb.ms_c2[m][j]]) * w;
                }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {   // first split in scan order among the minima
            float ov = __shfl_down_sync(0xffffffffu, bv, o);
            int oc = __shfl_down_sync(0xffffffffu, code, o);
            unsigned long long o1 = __shfl_down_sync(0xffffffffu, b1, o), o2 = __shfl_down_sync(0xffffffffu, b2, o);
            if (ov < bv || (ov == bv && oc < code)) { bv = ov; code = oc; b1 = o1; b2 = o2; }
        }
        if (lane == 0) {
            if (kept || code == 0x7fffffff) {
                unsigned long long li = atomicAdd(&ctr[0], 1ULL);
                if (li < cap) leaves[li] = nd; else ctr[1] = 1;
            } else if (depth >= 63) {
                ctr[1] = 1;
            } else {
                unsigned long long ni = atomicAdd(&ctr[2 + depth + 1], 2ULL);
                if (ni + 2 > cap) ctr[1] = 1;
                else {
                    nxt[ni].pat = b1;
                    nxt[ni].key = nd.key;
                    nxt[ni + 1].pat = b2;
                    nxt[ni + 1].key = nd.key | (1ULL << (63 - depth));
                }
            }
        }
    }
}

__global__ void __launch_bounds__(256) kp_backtrack_level_kernel(const KpTables *tab, const uint8_t *rowtab, const KpView vw,
                                                                 int depth, const KpBtNode *cur, KpBtNode *nxt,
                                                                 KpBtNode *leaves, unsigned long long cap,
                                                                 unsigned long long *ctr)
{
    kp_backtrack_level(*tab, rowtab, vw, depth, cur, nxt, leaves, cap, ctr, ctr[2 + depth]);
}

// All depths in one launch (cooperative launch: every CTA is resident), a grid-wide barrier between depths:
// ctr[72] counts arrivals.  Stops at the first empty frontier.
__global__ void __launch_bounds__(256) kp_backtrack_all_kernel(const KpTables *tab, const uint8_t *rowtab, const KpView vw,
                                                               int levels, KpBtNode *fa, KpBtNode *fb, KpBtNode *leaves,
                                                               unsigned long long cap, unsigned long long *ctr)
{
    const KpTables &tb = *tab;
    for (int d = 0; d < levels; d++) {
        const unsigned long long ncur = __ldcg(&ctr[2 + d]);
        if (ncur == 0) break;   // the same value in every CTA: it was final before the last barrier
        kp_backtrack_level(tb, rowtab, vw, d, (d & 1) ? fb : fa, (d & 1) ? fa : fb, leaves, cap, ctr, ncur < cap ? ncur : cap);
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) {
            atomicAdd(&ctr[72], 1ULL);
            const unsigned long long want = (unsigned long long)(d + 1) * gridDim.x;
            unsigned long long seen;
            do {
                asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(seen) : "l"(ctr + 72) : "memory");
                if (seen < want) __nanosleep(100);
            } while (seen < want);
        }
        __syncthreads();
    }
}

__global__ void kp_backtrack_init_kernel(KpBtNode *fa, unsigned long long top, unsigned long long *ctr)
{
    if (threadIdx.x < 80) ctr[threadIdx.x] = 0;
    __syncthreads();
    if (threadIdx.x == 0) { fa[0].pat = top; fa[0].key = 0; ctr[2] = 1; }
}

// rank sort by key (keys are distinct): out[rank] = pat
__global__ void kp_backtrack_sort_kernel(const KpBtNode *leaves, const unsigned long long *counts,
                                         unsigned long long cap, unsigned long long *out, unsigned long long *keys_out)
{
    unsigned long long n = counts[0];
    if (n > cap) n = cap;
    __shared__ unsigned long long keys[256];
    for (unsigned long long i0 = (unsigned long long)blockIdx.x * blockDim.x; i0 < n; i0 += (unsigned long long)gridDim.x * blockDim.x) {
        unsigned long long i = i0 + threadIdx.x;
        unsigned long long mykey = i < n ? leaves[i].key : 0, rank = 0;
        for (unsigned long long base = 0; base < n; base += 256) {
            unsigned long long j = base + threadIdx.x;
            keys[threadIdx.x] = j < n ? leaves[j].key : ~0ULL;
            __syncthreads();
            unsigned long long lim = n - base < 256 ? n - base : 256;
            for (unsigned long long t = 0; t < lim; t++) rank += keys[t] < mykey;
            __syncthreads();
        }
        if (i < n) { out[rank] = leaves[i].pat; keys_out[rank] = mykey; }
    }
}

// ---------------------------------------------------------------------------------------------------
// Greedy top-down partition (reference: greedy_penalty_plus_pseudo.py:155-196, greedy_res_kmer_table_ord).
// A node is a pattern; its loss is the float64 self-score of its counts; among all two-way splits of one position
// (scan order: string position, then split index) the first one whose float64 sum of the two children's losses is
// the strict minimum below the node's own loss is taken, and both children are expanded in turn.
// Two launches per depth.  The k-mers of a node are walked once, accumulating for every position and base the counts
// of the node restricted to that base (shared-memory atomics, then global ones); every candidate child is a sum of
// at most three of those marginals, so all candidates of the node are scored from that one pass.
// ---------------------------------------------------------------------------------------------------
struct KpGreedyLeaf { unsigned long long pat, key; double loss, test; };

// per-node accumulators in global memory: [position][base][M, U], then M, U, held-out M, held-out U of the node
#define KP_GREEDY_ACC (KP_MAXPOS * 8 + 4)

// Step 1 of a depth: marginal counts of every frontier node.  Small nodes: one CTA each.  Nodes with at least
// `big` k-mers (the first few depths): every CTA takes a slice.  Shared-memory atomics per CTA, then one global
// atomicAdd per non-zero counter.
__global__ void __launch_bounds__(256) kp_greedy_marginals_kernel(const KpTables *tab, const long long *kmerM, const long long *kmerU,
                                                                  const long long *testM, const long long *testU, int depth,
                                                                  const KpBtNode *cur, const unsigned long long *cur_size,
                                                                  const unsigned long long *ctr, unsigned long long big,
                                                                  unsigned long long *acc)
{
    const KpTables &tb = *tab;
    __shared__ unsigned long long marg[KP_GREEDY_ACC];
    __shared__ uint8_t s_bases[KP_MAXPOS][4];
    __shared__ uint32_t s_n[KP_MAXPOS];
    const unsigned long long ncur = ctr[2 + depth];
    const int npos = tb.npos;
    for (unsigned long long ni = 0; ni < ncur; ni++) {
        const unsigned long long total = cur_size[ni];   // k-mers of the node
        const bool shared_node = total >= big;
        if (!shared_node && ni % gridDim.x != blockIdx.x) continue;
        const KpBtNode nd = cur[ni];
        __syncthreads();   // previous node's readers are done
        if (threadIdx.x < npos) {
            const int e = threadIdx.x;
            const unsigned m = tb.digit_mask[e][(int)((nd.pat / tb.extw[e]) % tb.radix[e])];
            int n = 0;
            for (int b = 0; b < 4; b++)
                if ((m >> b) & 1u) s_bases[e][n++] = (uint8_t)b;
            s_n[e] = (uint32_t)n;
        }
        for (int i = threadIdx.x; i < KP_GREEDY_ACC; i += blockDim.x) marg[i] = 0;
        __syncthreads();
        unsigned long long aM = 0, aU = 0, aTM = 0, aTU = 0;
        const unsigned long long first = shared_node ? (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x : threadIdx.x;
        const unsigned long long step = shared_node ? (unsigned long long)gridDim.x * blockDim.x : blockDim.x;
        for (unsigned long long t = first; t < total; t += step) {
            unsigned long long r = t, kidx = 0;
            uint8_t pick[KP_MAXPOS];
            for (int e = 0; e < npos; e++) {
                const uint32_t n = s_n[e];
                const int b = s_bases[e][r % n];
                r /= n;
                pick[e] = (uint8_t)b;
                kidx += (unsigned long long)tb.mask_digit[e][1u << b] * tb.kw[e];
            }
            const unsigned long long M = (unsigned long long)kmerM[kidx], U = (unsigned long long)kmerU[kidx];
            aM += M; aU += U;
            if (testM) { aTM += (unsigned long long)testM[kidx]; aTU += (unsigned long long)testU[kidx]; }
            for (int e = 0; e < npos; e++)
                if (s_n[e] > 1) {
                    if (M) atomicAdd(&marg[(e * 4 + pick[e]) * 2 + 0], M);
                    if (U) atomicAdd(&marg[(e * 4 + pick[e]) * 2 + 1], U);
                }
        }
        if (aM) atomicAdd(&marg[KP_MAXPOS * 8 + 0], aM);
        if (aU) atomicAdd(&marg[KP_MAXPOS * 8 + 1], aU);
        if (aTM) atomicAdd(&marg[KP_MAXPOS * 8 + 2], aTM);
        if (aTU) atomicAdd(&marg[KP_MAXPOS * 8 + 3], aTU);
        __syncthreads();
        for (int i = threadIdx.x; i < KP_GREEDY_ACC; i += blockDim.x)
            if (marg[i]) atomicAdd(&acc[ni * KP_GREEDY_ACC + i], marg[i]);
    }
}

// Step 2 of a depth: one warp per node scores the node and every candidate split from the marginals, decides, and
// clears the node's accumulators for the next depth.
__global__ void __launch_bounds__(256) kp_greedy_decide_kernel(const KpTables *tab, int has_test, double alpha, double beta,
                                                               double penalty, int depth, const KpBtNode *cur,
                                                               const unsigned long long *cur_size, KpBtNode *nxt,
                                                               unsigned long long *nxt_size, KpGreedyLeaf *leaves,
                                                               unsigned long long cap, unsigned long long *ctr,
                                                               unsigned long long *acc)
{
    const KpTables &tb = *tab;
    __shared__ double2 logtab[128];
    for (int i = threadIdx.x; i < 128; i += blockDim.x) logtab[i] = make_double2(kpc_logTab[2 * i], kpc_logTab[2 * i + 1]);
    __syncthreads();
    const KpLogK K = kp_logk_load();
    const unsigned long long ncur = ctr[2 + depth];
    const int npos = tb.npos, lane = threadIdx.x & 31;
    const unsigned long long nw = (unsigned long long)gridDim.x * (blockDim.x >> 5);
    for (unsigned long long ni = (unsigned long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); ni < ncur; ni += nw) {
        const KpBtNode nd = cur[ni];
        unsigned long long *marg = acc + ni * KP_GREEDY_ACC;
        const unsigned long long tM = marg[KP_MAXPOS * 8 + 0], tU = marg[KP_MAXPOS * 8 + 1];
        const unsigned long long hM = marg[KP_MAXPOS * 8 + 2], hU = marg[KP_MAXPOS * 8 + 3];
        double lp0, l10;
        const double self = kp_self_score_t<unsigned long long>(tM, tU, alpha, beta, penalty, logtab, K, lp0, l10);
        // candidates in scan order: (position e, split j) -> rank pos_id[e] * 8 + j
        double bv = self;
        int brank = 0x7fffffff;
        unsigned long long b1 = 0, b2 = 0, z1 = 0, z2 = 0;   // children and their sizes
        const unsigned long long mysize = cur_size[ni];
        int c = 0;
        for (int e = 0; e < npos; e++) {
            const int d = (int)((nd.pat / tb.extw[e]) % tb.radix[e]);
            const unsigned m = tb.digit_mask[e][d];
            const int ns = tb.ms_n[m];
            for (int j = 0; j < ns; j++, c++) {
                if ((c & 31) != lane) continue;
                const unsigned m1 = tb.ms_c1[m][j], m2 = tb.ms_c2[m][j];
                unsigned long long M1 = 0, U1 = 0, M2 = 0, U2 = 0;
                for (int b = 0; b < 4; b++) {
                    if ((m1 >> b) & 1u) { M1 += marg[(e * 4 + b) * 2]; U1 += marg[(e * 4 + b) * 2 + 1]; }
                    if ((m2 >> b) & 1u) { M2 += marg[(e * 4 + b) * 2]; U2 += marg[(e * 4 + b) * 2 + 1]; }
                }
                double lpa, l1a;
                const double s1 = kp_self_score_t<unsigned long long>(M1, U1, alpha, beta, penalty, logtab, K, lpa, l1a);
                const double s2 = kp_self_score_t<unsigned long long>(M2, U2, alpha, beta, penalty, logtab, K, lpa, l1a);
                const double sum = KP_ADD(s1, s2);
                if (sum < bv) {   // within a lane the ranks only grow: a later equal sum never replaces an earlier one
                    bv = sum;
                    brank = tb.pos_id[e] * 8 + j;
                    b1 = nd.pat - (unsigned long long)(d - (int)tb.mask_digit[e][m1]) * tb.extw[e];
                    b2 = nd.pat - (unsigned long long)(d - (int)tb.mask_digit[e][m2]) * tb.extw[e];
                    z1 = mysize / (unsigned)__popc(m) * (unsigned)__popc(m1);
                    z2 = mysize / (unsigned)__popc(m) * (unsigned)__popc(m2);
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {   // strict minimum below the node's loss, earliest in scan order among equals
            const double ov = __shfl_down_sync(0xffffffffu, bv, o);
            const int orank = __shfl_down_sync(0xffffffffu, brank, o);
            const unsigned long long o1 = __shfl_down_sync(0xffffffffu, b1, o), o2 = __shfl_down_sync(0xffffffffu, b2, o);
            const unsigned long long y1 = __shfl_down_sync(0xffffffffu, z1, o), y2 = __shfl_down_sync(0xffffffffu, z2, o);
            if (orank != 0x7fffffff && (ov < bv || (ov == bv && orank < brank))) {
                bv = ov; brank = orank; b1 = o1; b2 = o2; z1 = y1; z2 = y2;
            }
        }
        __syncwarp();
        for (int i = lane; i < KP_GREEDY_ACC; i += 32) marg[i] = 0;   // clean for the next depth
        if (lane == 0) {
            if (brank == 0x7fffffff) {   // no split beats the node: a leaf of the partition
                const unsigned long long li = atomicAdd(&ctr[0], 1ULL);
                if (li < cap) {
                    KpGreedyLeaf L;
                    L.pat = nd.pat; L.key = nd.key; L.loss = self;
                    L.test = has_test ? kp_test_ll_t<unsigned long long>(hM, hU, lp0, l10) : 0.0;
                    leaves[li] = L;
                } else ctr[1] = 1;
            } else if (depth >= 63) {
                ctr[1] = 1;
            } else {
                const unsigned long long q = atomicAdd(&ctr[2 + depth + 1], 2ULL);
                if (q + 2 > cap) ctr[1] = 1;
                else {
                    nxt[q].pat = b1; nxt[q].key = nd.key;
                    nxt[q + 1].pat = b2; nxt[q + 1].key = nd.key | (1ULL << (63 - depth));
                    nxt_size[q] = z1;
                    nxt_size[q + 1] = z2;
                }
            }
        }
    }
}

__global__ void kp_greedy_init_kernel(unsigned long long *size0, unsigned long long nkmer) { size0[0] = nkmer; }

// rank sort of the greedy leaves by path key (depth-first, first child first): out[rank] = leaf
__global__ void kp_greedy_sort_kernel(const KpGreedyLeaf *leaves, const unsigned long long *counts, unsigned long long cap,
                                      KpGreedyLeaf *out)
{
    unsigned long long n = counts[0];
    if (n > cap) n = cap;
    __shared__ unsigned long long keys[256];
    for (unsigned long long i0 = (unsigned long long)blockIdx.x * blockDim.x; i0 < n; i0 += (unsigned long long)gridDim.x * blockDim.x) {
        unsigned long long i = i0 + threadIdx.x;
        unsigned long long mykey = i < n ? leaves[i].key : 0, rank = 0;
        for (unsigned long long base = 0; base < n; base += 256) {
            unsigned long long j = base + threadIdx.x;
            keys[threadIdx.x] = j < n ? leaves[j].key : ~0ULL;
            __syncthreads();
            unsigned long long lim = n - base < 256 ? n - base : 256;
            for (unsigned long long t = 0; t < lim; t++) rank += keys[t] < mykey;
            __syncthreads();
        }
        if (i < n) out[rank] = leaves[i];
    }
}

// split codes of arbitrary patterns (test hook and output stage)
__global__ void kp_split_codes_kernel(const KpTables *tab, const uint8_t *rowtab, const KpView vw,
                                      const unsigned long long *pats, unsigned long long n, uint8_t *codes)
{
    const KpTables &tb = *tab;
    const uint16_t *srow_of_row = (const uint16_t *)(rowtab + tb.rt_srow_of_row);
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        unsigned long long p1, p2;
        codes[i] = kp_split_code_dev(tb, srow_of_row, vw, pats[i], &p1, &p2);
    }
}

// gather table values of arbitrary patterns: out[i] = table[pattern i]  (also: unpacks whole tables for tests)
__global__ void kp_gather_kernel(const KpTables *tab, const uint8_t *rowtab, const KpView vw,
                                 const unsigned long long *pats, unsigned long long first, unsigned long long n, float *out)
{
    const KpTables &tb = *tab;
    const uint16_t *srow_of_row = (const uint16_t *)(rowtab + tb.rt_srow_of_row);
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x)
        out[i] = kp_best_at(tb, srow_of_row, vw, pats ? pats[i] : first + i);
}

__global__ void kp_gather_flags_kernel(const KpTables *tab, const uint8_t *rowtab, const KpView vw,
                                       const unsigned long long *pats, unsigned long long first, unsigned long long n, uint8_t *out)
{
    const KpTables &tb = *tab;
    const uint16_t *srow_of_row = (const uint16_t *)(rowtab + tb.rt_srow_of_row);
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        KpLoc L = kp_locate_dev(tb, srow_of_row, pats ? pats[i] : first + i);
        out[i] = (uint8_t)kp_view_kept(tb, vw, L.tile, L.srow, L.d0);
    }
}

// ---------------------------------------------------------------------------------------------------
// counts of arbitrary patterns from the k-mer tables: one CTA per pattern at a time, and the CTA enumerates only the
// k-mers the pattern matches (mixed radix over the sizes of its per-position subsets), so a whole partition costs
// one pass over the 4^k k-mers (pattern_utils.py:192-215 walks matches() the same way, in Python)
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) kp_pattern_counts_kernel(const KpTables *tab, unsigned long long npatq,
                                                                const long long *kmerM, const long long *kmerU,
                                                                const unsigned long long *patnums, long long *outM,
                                                                long long *outU)
{
    const KpTables &tb = *tab;
    __shared__ uint32_t s_n[KP_MAXPOS];          // bases in the subset of position e
    __shared__ uint32_t s_off[KP_MAXPOS][4];     // k-mer index contribution of each of them
    __shared__ unsigned long long s_total;
    __shared__ long long redM[256], redU[256];
    for (unsigned long long q = blockIdx.x; q < npatq; q += gridDim.x) {
        if (threadIdx.x == 0) {
            unsigned long long x = patnums[q], total = 1;
            for (int e = 0; e < tb.npos; e++) {
                const uint32_t m = tb.digit_mask[e][x % tb.radix[e]];
                x /= tb.radix[e];
                uint32_t n = 0;
                for (int b = 0; b < 4; b++)
                    if ((m >> b) & 1u) s_off[e][n++] = (uint32_t)tb.mask_digit[e][1u << b] * tb.kw[e];
                s_n[e] = n;
                total *= n;
            }
            s_total = total;
        }
        __syncthreads();
        long long am = 0, au = 0;
        const unsigned long long total = s_total;
        for (unsigned long long j = threadIdx.x; j < total; j += blockDim.x) {
            unsigned long long r = j;
            uint32_t kidx = 0;
            for (int e = 0; e < tb.npos; e++) {
                const uint32_t n = s_n[e];
                kidx += s_off[e][r % n];
                r /= n;
            }
            am += kmerM[kidx];
            au += kmerU[kidx];
        }
        redM[threadIdx.x] = am; redU[threadIdx.x] = au;
        __syncthreads();
        for (int s = 128; s > 0; s >>= 1) {
            if ((int)threadIdx.x < s) { redM[threadIdx.x] += redM[threadIdx.x + s]; redU[threadIdx.x] += redU[threadIdx.x + s]; }
            __syncthreads();
        }
        if (threadIdx.x == 0) { outM[q] = redM[0]; outU[q] = redU[0]; }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------
// test hooks
// ---------------------------------------------------------------------------------------------------
__global__ void kp_debug_log_kernel(const double *x, double *y, unsigned long long n)
{
    __shared__ double2 tab[128];
    for (int i = threadIdx.x; i < 128; i += blockDim.x) tab[i] = make_double2(kpc_logTab[2 * i], kpc_logTab[2 * i + 1]);
    __syncthreads();
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x)
        y[i] = kp_log(x[i], tab);
}

// per-(k-mer, fold) terms of the all-k-mers model (all_kmers_CV.py:8-13, :42-43): the level-0 formulas with no penalty
__global__ void kp_kmer_fold_terms_kernel(const long long *Mtr, const long long *Utr, const long long *Mte, const long long *Ute,
                                          const double *beta, unsigned long long n, double alpha, double *train, double *test)
{
    __shared__ double2 tab[128];
    for (int i = threadIdx.x; i < 128; i += blockDim.x) tab[i] = make_double2(kpc_logTab[2 * i], kpc_logTab[2 * i + 1]);
    __syncthreads();
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        double a, b;
        kp_leaf_cv((unsigned long long)Mtr[i], (unsigned long long)Utr[i], (unsigned long long)Mte[i], (unsigned long long)Ute[i],
                   alpha, beta[i], 0.0, tab, a, b);
        train[i] = a;
        test[i] = b;
    }
}

__global__ void kp_debug_leaf_kernel(const long long *M, const long long *U, unsigned long long n, double alpha,
                                     double beta, double penalty, double *out)
{
    __shared__ double2 tab[128];
    for (int i = threadIdx.x; i < 128; i += blockDim.x) tab[i] = make_double2(kpc_logTab[2 * i], kpc_logTab[2 * i + 1]);
    __syncthreads();
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x)
        out[i] = kp_leaf_score((unsigned long long)M[i], (unsigned long long)U[i], alpha, beta, penalty, tab);
}

// The three level >= 1 scoring paths of the DP kernels for one item: the score filter's lower bound (per-base counts
// converted to float and summed in base order, as the kernels do), the fast score (ok, sf, rounded-up bit, s~) and the
// exact score, in the count width C.  M, U: [n][4] per-base counts.
template <typename C>
__device__ void kp_debug_self_score_one(const long long *M, const long long *U, double alpha, double beta, double penalty,
                                        const double2 *tab, float &lb, unsigned char &ok, float &sf, unsigned char &rup,
                                        double &st, double &exact)
{
    C m[4], u[4], M_ = 0, U_ = 0;
    float2 Mf = make_float2(0.f, 0.f), Uf = make_float2(0.f, 0.f);
    for (int b = 0; b < 4; b++) {
        m[b] = (C)M[b];
        u[b] = (C)U[b];
        M_ += m[b];
        U_ += u[b];
        Mf.x += (float)m[b];
        Uf.x += (float)u[b];
    }
    Mf.y = Mf.x;
    Uf.y = Uf.x;
    lb = kp_score_lower_bound2(Mf, Uf, kp_filter_consts(alpha, beta, penalty)).x;
    const KpLogK K = kp_logk_load();
    bool r = false;
    ok = kp_self_score_fast<C>(M_, U_, alpha, beta, penalty, tab, K, sf, r, &st);
    rup = r;
    exact = kp_self_score_exact_nl<C>(M_, U_, alpha, beta, penalty, tab);
}

__global__ void kp_debug_self_score_kernel(const long long *M, const long long *U, const double *alpha, const double *beta,
                                           const double *penalty, const unsigned char *wide, unsigned long long n, float *lb,
                                           unsigned char *ok, float *sf, unsigned char *rup, double *st, double *exact)
{
    __shared__ double2 tab[128];
    for (int i = threadIdx.x; i < 128; i += blockDim.x) tab[i] = make_double2(kpc_logTab[2 * i], kpc_logTab[2 * i + 1]);
    __syncthreads();
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        if (wide[i])
            kp_debug_self_score_one<unsigned long long>(M + 4 * i, U + 4 * i, alpha[i], beta[i], penalty[i], tab, lb[i], ok[i],
                                                        sf[i], rup[i], st[i], exact[i]);
        else
            kp_debug_self_score_one<unsigned int>(M + 4 * i, U + 4 * i, alpha[i], beta[i], penalty[i], tab, lb[i], ok[i], sf[i],
                                                  rup[i], st[i], exact[i]);
    }
}
