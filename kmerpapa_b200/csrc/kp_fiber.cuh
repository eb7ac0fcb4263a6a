// kp_fiber.cuh — K3+K4 with a FOURTH position on chip (sm_100a).
//
// kp_dp_rows_kernel (kp_kernels.cuh) keeps three N positions of a tile on chip and streams the two child tiles of every
// split of the five remaining ("high") positions from HBM/L2: 16.7 child-tile reads per tile written.  Here one of the
// high positions, the FIBER position, comes on chip too: a CTA owns the 15 tiles that differ only in that digit
// (a fiber: 15^4 = 50 625 patterns, 202.5 KB of float32, almost all of the SM's 227 KB of shared memory), so only the
// splits of the other high positions are streamed: 13.3 child-tile reads per tile, one fifth fewer bytes through L2 and
// HBM.  Waves run over the fibers (level of the other high positions): 13 launches for NNNNANNNN instead of 16.
//
// Per fiber, the whole CTA (16 warps):
//   1. lists the fiber's high splits (the same for its 15 tiles: a child fiber is the parent fiber moved along one
//      other position) and loads the 15 x 64 base k-mer counts;
//   2. STREAM: for every float4 of the fiber, min over the splits of (child1 + child2), loads batched 2 x 4 x 2 LDG.128
//      per thread (128 KB in flight per SM), straight from registers into the shared-memory copy of the fiber;
//   3. LEVELS: the 15 x 225 rows are visited in 10 steps by level(fiber digit) + level(row); one lane owns one row (its
//      15 sub-patterns of the register position in registers): splits of the fiber position and cross-row splits
//      from shared memory, row counts, score filter, exact float64 score for the survivors, in-register splits -
//      the same arithmetic as kp_dp_rows_kernel, statement for statement, so the tables are bit-identical;
//   4. copies the finished fiber out with coalesced 16-byte stores (HBM layout unchanged: schedule-order rows).
// The rows of a tile sit in LEVEL order in shared memory (lanes of a warp then read consecutive 16-byte slots: no bank
// conflicts); the 16th (padding) slot of a row is not kept on chip: groups 0-2 are float4 planes, group 3 three float
// planes.
#pragma once
#include "kp_kernels.cuh"

#define KP_FIBER_THREADS 512
#define KP_FIBER_CELLS (KP_FIBER_DIGITS * KP_FIBER_ROWS)   // rows of a fiber: 3375

struct KpFiberParams {
    const KpTables *tab;
    const KpFiberTables *ftab;
    const uint8_t *fiberblob;
    const uint32_t *fiber_list;  // fibers of this wave (tile id of the digit-0 tile), ascending
    uint32_t nfibers_wave;
    uint32_t *counter;           // next unclaimed entry of fiber_list (zeroed before the launch)
    int leaf_wave;               // wave 0: tiles whose fiber digit is a single nucleotide hold k-mers in their level-0 rows
    const long long *e0, *e1;    // expanded counts M, U  [ntiles][tile_kmers]
    const long long *s0, *s1;    // CV job: held-out expanded counts, subtracted on the fly; else null
    double alpha, beta, penalty;
    float *best;
    uint16_t *flags;
    int dbg;                     // timing experiments only (KP_FIBER_DBG): 1 = skip the stream phase, 2 = skip the level phase
};

// shared-memory map of the fiber kernel (bytes)
struct KpFiberSmem {
    uint32_t logtab, blob, bc, hs, misc, fsplit, flags, planes, total;
};

__host__ __device__ inline KpFiberSmem kp_fiber_smem(uint32_t ft_bytes, uint32_t maxhs, uint32_t tile_kmers, bool wide)
{
    KpFiberSmem m;
    uint32_t o = 0;
    m.logtab = o; o += 2048;
    m.blob = o; o += (ft_bytes + 15u) & ~15u;
    m.bc = o; o += KP_FIBER_DIGITS * tile_kmers * 2u * (wide ? 8u : 4u);
    m.hs = o; o += ((maxhs * 8u) + 15u) & ~15u;
    m.misc = o; o += 256;
    m.fsplit = o; o += 256;
    m.flags = o; o += (KP_FIBER_CELLS * 2u + 15u) & ~15u;
    m.planes = o; o += KP_FIBER_CELLS * 60u;
    m.total = o;
    return m;
}

// the 15 values of a row in the shared-memory planes
struct KpFiberS {
    float4 *P0, *P1, *P2;
    float *Q0, *Q1, *Q2;
    __device__ __forceinline__ void load(int idx, float *v) const
    {
        const float4 a = P0[idx], b = P1[idx], c = P2[idx];
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
        v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
        v[8] = c.x; v[9] = c.y; v[10] = c.z; v[11] = c.w;
        v[12] = Q0[idx]; v[13] = Q1[idx]; v[14] = Q2[idx];
    }
    __device__ __forceinline__ void store(int idx, const float *v) const
    {
        P0[idx] = make_float4(v[0], v[1], v[2], v[3]);
        P1[idx] = make_float4(v[4], v[5], v[6], v[7]);
        P2[idx] = make_float4(v[8], v[9], v[10], v[11]);
        Q0[idx] = v[12]; Q1[idx] = v[13]; Q2[idx] = v[14];
    }
};

// v = min(v, a + b) over the 15 cells of two rows in shared memory (packed f32x2 adds, IEEE round-to-nearest)
__device__ __forceinline__ void kp_fiber_split1(const KpFiberS &S, int ia, int ib, float *v)
{
    float xa[16], xb[16];
    S.load(ia, xa);
    S.load(ib, xb);
#pragma unroll
    for (int c = 0; c < 14; c += 2) {
        const float2 s = __fadd2_rn(make_float2(xa[c], xa[c + 1]), make_float2(xb[c], xb[c + 1]));
        v[c] = fminf(v[c], s.x);
        v[c + 1] = fminf(v[c + 1], s.y);
    }
    v[14] = fminf(v[14], __fadd_rn(xa[14], xb[14]));
}

// two splits per pass: one 3-input min per cell
__device__ __forceinline__ void kp_fiber_split2(const KpFiberS &S, int ia, int ib, int ic, int ie, float *v)
{
    float xa[16], xb[16], xc[16], xe[16];
    S.load(ia, xa);
    S.load(ib, xb);
    S.load(ic, xc);
    S.load(ie, xe);
#pragma unroll
    for (int c = 0; c < 14; c += 2) {
        const float2 s1 = __fadd2_rn(make_float2(xa[c], xa[c + 1]), make_float2(xb[c], xb[c + 1]));
        const float2 s2 = __fadd2_rn(make_float2(xc[c], xc[c + 1]), make_float2(xe[c], xe[c + 1]));
        v[c] = kp_min3(v[c], s1.x, s2.x);
        v[c + 1] = kp_min3(v[c + 1], s1.y, s2.y);
    }
    v[14] = kp_min3(v[14], __fadd_rn(xa[14], xb[14]), __fadd_rn(xc[14], xe[14]));
}

__device__ __forceinline__ float4 kp_min4(float4 m, float4 a, float4 b)
{
    const float2 lo = __fadd2_rn(make_float2(a.x, a.y), make_float2(b.x, b.y));
    const float2 hi = __fadd2_rn(make_float2(a.z, a.w), make_float2(b.z, b.w));
    return make_float4(fminf(m.x, lo.x), fminf(m.y, lo.y), fminf(m.z, hi.x), fminf(m.w, hi.y));
}

template <bool WIDE>
__global__ void __launch_bounds__(KP_FIBER_THREADS, 1) kp_dp_fiber_kernel(const KpFiberParams p)
{
    typedef typename KpCnt<WIDE>::type C;
    constexpr int R0 = 15, NB = 4, NT = KP_FIBER_THREADS, NR = KP_FIBER_ROWS, RP = 232;
    constexpr int TILE4 = 4 * RP;                       // float4 per tile in HBM
    constexpr int NJ = KP_FIBER_DIGITS * TILE4;         // float4 per fiber in HBM (padding included)

    extern __shared__ __align__(16) unsigned char smem[];
    const KpTables &tb = *p.tab;
    const KpFiberTables &ft = *p.ftab;
    const int tid = threadIdx.x;
    const uint32_t tk = tb.tile_kmers;
    const KpFiberSmem sm = kp_fiber_smem(ft.ft_bytes, ft.maxhs, tk, WIDE);

    double2 *logtab = (double2 *)(smem + sm.logtab);
    unsigned char *blob = smem + sm.blob;
    C *bc = (C *)(smem + sm.bc);                        // [15][tile_kmers][2]
    uint32_t *hs1 = (uint32_t *)(smem + sm.hs), *hs2 = hs1 + ft.maxhs;
    int *misc = (int *)(smem + sm.misc);                // [0] fiber index claimed, [1] number of high splits, [8..] level tables
    uint8_t *fsplit = smem + sm.fsplit;                 // [15][8][2] child digits of the fiber-position splits; [240 + d] their number
    uint16_t *sflags = (uint16_t *)(smem + sm.flags);
    KpFiberS S;
    S.P0 = (float4 *)(smem + sm.planes);
    S.P1 = S.P0 + KP_FIBER_CELLS;
    S.P2 = S.P1 + KP_FIBER_CELLS;
    S.Q0 = (float *)(S.P2 + KP_FIBER_CELLS);
    S.Q1 = S.Q0 + KP_FIBER_CELLS;
    S.Q2 = S.Q1 + KP_FIBER_CELLS;

    for (int i = tid; i < 128; i += NT) logtab[i] = make_double2(kpc_logTab[2 * i], kpc_logTab[2 * i + 1]);
    for (uint32_t i = tid; i < ft.ft_bytes / 4; i += NT) ((uint32_t *)blob)[i] = ((const uint32_t *)p.fiberblob)[i];
    if (tid < KP_FIBER_DIGITS) {   // splits of the fiber position, as digit pairs
        const int e = ft.fe, d = tid;
        const uint32_t m = tb.digit_mask[e][d];
        const int ns = tb.ms_n[m];
        for (int j = 0; j < ns; j++) {
            fsplit[(d * 8 + j) * 2 + 0] = tb.mask_digit[e][tb.ms_c1[m][j]];
            fsplit[(d * 8 + j) * 2 + 1] = tb.mask_digit[e][tb.ms_c2[m][j]];
        }
        fsplit[240 + d] = (uint8_t)ns;
    }
    __syncthreads();
    const uint8_t *frow_of_srow = blob + ft.ft_frow_of_srow;
    const uint16_t *xs_off = (const uint16_t *)(blob + ft.ft_xs_off);
    const uint16_t *xs = (const uint16_t *)(blob + ft.ft_xs);
    const uint16_t *bs_off = (const uint16_t *)(blob + ft.ft_bs_off);
    const uint8_t *bs = blob + ft.ft_bs;
    uint32_t lvl_start[KP_FIBER_ROW_LEVELS + 1];
#pragma unroll
    for (int l = 0; l <= KP_FIBER_ROW_LEVELS; l++) lvl_start[l] = ft.lvl_start[l];

    const double alpha = p.alpha, beta = p.beta, penalty = p.penalty;
    const KpFilterK fk = kp_filter_consts(alpha, beta, penalty);
    const float INF = __int_as_float(0x7f800000);
    const uint32_t hwf = ft.hw;
    const int nhigh = tb.nhigh, fhi = ft.fhi;
    const float4 *tb4 = (const float4 *)p.best;

    for (;;) {
        __syncthreads();   // the previous fiber has left shared memory
        if (tid == 0) misc[0] = (int)atomicAdd(p.counter, 1u);
        // ---- the fiber's high-position splits (two child fibers each), by warp 0 ----
        __syncthreads();
        const uint32_t it = (uint32_t)misc[0];
        if (it >= p.nfibers_wave) break;
        const uint32_t base = p.fiber_list[it];
        if (tid < 32) {
            int ns = 0, d = 0, e = 0;
            uint32_t m = 0, hw = 1;
            if (tid < nhigh && tid != fhi) {
                e = tb.highpos[tid];
                hw = tb.highw[e];
                d = (int)((base / hw) % tb.radix[e]);
                m = tb.digit_mask[e][d];
                ns = tb.ms_n[m];
            }
            int off = ns;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int x = __shfl_up_sync(0xffffffffu, off, o);
                if (tid >= o) off += x;
            }
            const int total = __shfl_sync(0xffffffffu, off, 31);
            off -= ns;
            for (int j = 0; j < ns; j++) {
                const int c1 = tb.mask_digit[e][tb.ms_c1[m][j]], c2 = tb.mask_digit[e][tb.ms_c2[m][j]];
                hs1[off + j] = base - (uint32_t)(d - c1) * hw;
                hs2[off + j] = base - (uint32_t)(d - c2) * hw;
            }
            if (tid == 0) misc[1] = total;
        }
        // ---- base counts of the 15 tiles ----
        for (uint32_t i = tid; i < KP_FIBER_DIGITS * tk; i += NT) {
            const uint32_t x = i / tk, kl = i - x * tk;
            const size_t g = (size_t)(base + x * hwf) * tk + kl;
            bc[i * 2 + 0] = (C)(p.s0 ? p.e0[g] - p.s0[g] : p.e0[g]);
            bc[i * 2 + 1] = (C)(p.s1 ? p.e1[g] - p.s1[g] : p.e1[g]);
        }
        __syncthreads();
        const int nhs = misc[1];

        // ---- STREAM: S = min over the high splits of (child fiber 1 + child fiber 2), for the whole fiber ----
        for (int j0 = tid; j0 < ((p.dbg & 1) ? 0 : NJ); j0 += 2 * NT) {
            const int j1 = j0 + NT;
            const int x0 = j0 / TILE4, r0 = j0 - x0 * TILE4;          // r = group * RP + srow
            const int x1 = j1 / TILE4, r1 = j1 - x1 * TILE4;
            const int g0 = r0 / RP, srow0 = r0 - g0 * RP;
            const int g1 = r1 / RP, srow1 = r1 - g1 * RP;
            const bool ok0 = srow0 < NR, ok1 = j1 < NJ && srow1 < NR;
            const size_t o0 = (size_t)x0 * hwf * TILE4 + r0, o1 = (size_t)x1 * hwf * TILE4 + r1;
            float4 acc0 = make_float4(INF, INF, INF, INF), acc1 = acc0;
            for (int s0 = 0; s0 < nhs; s0 += 4) {
                float4 a0[4], b0[4], a1[4], b1[4];
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    a0[q] = b0[q] = a1[q] = b1[q] = make_float4(INF, INF, INF, INF);
                    if (s0 + q < nhs) {
                        const float4 *c1 = tb4 + (size_t)hs1[s0 + q] * TILE4, *c2 = tb4 + (size_t)hs2[s0 + q] * TILE4;
                        if (ok0) { a0[q] = __ldg(c1 + o0); b0[q] = __ldg(c2 + o0); }
                        if (ok1) { a1[q] = __ldg(c1 + o1); b1[q] = __ldg(c2 + o1); }
                    }
                }
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    acc0 = kp_min4(acc0, a0[q], b0[q]);
                    acc1 = kp_min4(acc1, a1[q], b1[q]);
                }
            }
            if (ok0) {
                const int idx = x0 * NR + frow_of_srow[srow0];
                if (g0 == 0) S.P0[idx] = acc0;
                else if (g0 == 1) S.P1[idx] = acc0;
                else if (g0 == 2) S.P2[idx] = acc0;
                else { S.Q0[idx] = acc0.x; S.Q1[idx] = acc0.y; S.Q2[idx] = acc0.z; }
            }
            if (ok1) {
                const int idx = x1 * NR + frow_of_srow[srow1];
                if (g1 == 0) S.P0[idx] = acc1;
                else if (g1 == 1) S.P1[idx] = acc1;
                else if (g1 == 2) S.P2[idx] = acc1;
                else { S.Q0[idx] = acc1.x; S.Q1[idx] = acc1.y; S.Q2[idx] = acc1.z; }
            }
        }
        __syncthreads();

        // ---- LEVELS: rows (fiber digit x, row) with level(x) + level(row) = L are independent ----
        for (int L = 0; L <= ((p.dbg & 2) ? -1 : 3 + KP_FIBER_ROW_LEVELS - 1); L++) {
            // the (up to four) groups of this level: digit level lx = 0..3 with row level L - lx
            int gstart[5];
            gstart[0] = 0;
#pragma unroll
            for (int lx = 0; lx < 4; lx++) {
                const int lr = L - lx;
                const int nx = lx == 0 ? 4 : (lx == 1 ? 6 : (lx == 2 ? 4 : 1));
                int nr = 0;
#pragma unroll
                for (int l = 0; l < KP_FIBER_ROW_LEVELS; l++)
                    if (l == lr) nr = (int)(lvl_start[l + 1] - lvl_start[l]);
                gstart[lx + 1] = gstart[lx] + nx * nr;
            }
            for (int k = tid; k < gstart[4]; k += NT) {
                const int lx = k < gstart[1] ? 0 : (k < gstart[2] ? 1 : (k < gstart[3] ? 2 : 3));
                const int lr = L - lx;
                const int xbase = lx == 0 ? 0 : (lx == 1 ? 4 : (lx == 2 ? 10 : 14));
                int rstart = 0, nr = 1;
#pragma unroll
                for (int l = 0; l < KP_FIBER_ROW_LEVELS; l++)
                    if (l == lr) { rstart = (int)lvl_start[l]; nr = (int)(lvl_start[l + 1] - lvl_start[l]); }
                const int kk = k - gstart[lx];
                const int xi = kk / nr;
                const int x = xbase + xi, frow = rstart + (kk - xi * nr);
                const int idx = x * NR + frow;

                float v[16];
                S.load(idx, v);   // minimum over the high-position splits, parked by the stream phase
                v[15] = INF;
                // ---- splits of the fiber position: the same row of two other tiles of the fiber ----
                {
                    const int nfs = fsplit[240 + x];
                    const uint8_t *fs = fsplit + x * 16;
                    int j = 0;
                    for (; j + 2 <= nfs; j += 2)
                        kp_fiber_split2(S, fs[2 * j] * NR + frow, fs[2 * j + 1] * NR + frow, fs[2 * j + 2] * NR + frow,
                                        fs[2 * j + 3] * NR + frow, v);
                    if (j < nfs) kp_fiber_split1(S, fs[2 * j] * NR + frow, fs[2 * j + 1] * NR + frow, v);
                }
                // ---- cross-row splits: finished rows of the same tile ----
                {
                    int i = xs_off[frow];
                    const int iend = xs_off[frow + 1];
                    const int xb = x * NR;
                    for (; i + 2 <= iend; i += 2) {
                        const uint32_t pr = xs[i], pq = xs[i + 1];
                        kp_fiber_split2(S, xb + (int)(pr & 0xFFu), xb + (int)(pr >> 8), xb + (int)(pq & 0xFFu), xb + (int)(pq >> 8), v);
                    }
                    if (i < iend) {
                        const uint32_t pr = xs[i];
                        kp_fiber_split1(S, xb + (int)(pr & 0xFFu), xb + (int)(pr >> 8), v);
                    }
                }
                // ---- counts of this row at the single-nucleotide digits of the register position ----
                C m[NB], u[NB];
#pragma unroll
                for (int b = 0; b < NB; b++) { m[b] = 0; u[b] = 0; }
                {
                    const C *bcx = bc + (size_t)x * tk * 2;
                    for (int i = bs_off[frow]; i < bs_off[frow + 1]; i++) {
                        const C *q = bcx + (size_t)bs[i] * NB * 2;
                        if (!WIDE) {
#pragma unroll
                            for (int b = 0; b < NB; b += 2) {
                                const uint4 y = *(const uint4 *)(q + b * 2);
                                m[b] += y.x; u[b] += y.y; m[b + 1] += y.z; u[b + 1] += y.w;
                            }
                        } else {
#pragma unroll
                            for (int b = 0; b < NB; b++) { m[b] += q[b * 2 + 0]; u[b] += q[b * 2 + 1]; }
                        }
                    }
                }
                // ---- score filter: which patterns can still be kept whole? (v only decreases from here) ----
                const bool leafrow = p.leaf_wave != 0 && lx == 0 && lr == 0;
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
                float sfx[16];
#pragma unroll
                for (int c = 0; c < 16; c++) sfx[c] = 0.f;
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
#pragma unroll
                        for (int c = 0; c < R0; c++)
                            if (c == d) sfx[c] = sf;
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
#undef KP_FIN
#undef KP_SP
#undef KP_SP2
                S.store(idx, v);
                sflags[idx] = (uint16_t)flag;
            }
            __syncthreads();
        }

        // ---- copy the fiber out: coalesced 16-byte stores in the HBM layout (schedule-order rows, 16 slots per row) ----
        for (int j = tid; j < NJ; j += NT) {
            const int x = j / TILE4, r = j - x * TILE4;
            const int g = r / RP, srow = r - g * RP;
            if (srow >= NR) continue;
            const int idx = x * NR + frow_of_srow[srow];
            float4 o;
            if (g == 0) o = S.P0[idx];
            else if (g == 1) o = S.P1[idx];
            else if (g == 2) o = S.P2[idx];
            else o = make_float4(S.Q0[idx], S.Q1[idx], S.Q2[idx], 0.f);
            __stcs((float4 *)p.best + (size_t)(base + x * hwf) * TILE4 + r, o);   // next read is a whole wave away
        }
        for (int j = tid; j < KP_FIBER_DIGITS * RP; j += NT) {
            const int x = j / RP, srow = j - x * RP;
            if (srow < NR) p.flags[(size_t)(base + x * hwf) * RP + srow] = sflags[x * NR + frow_of_srow[srow]];
        }
    }
}
