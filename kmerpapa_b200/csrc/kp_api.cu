// kp_api.cu — C ABI of libkpapa.so (see include/kmerpapa_b200.h for the contract).
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/kmerpapa_b200.h"
#include "kp_kernels.cuh"
#include "kp_fiber.cuh"
#include "kp_plan.h"
#include "kp_shard_owners.h"

namespace {

thread_local std::string g_err;

int fail(const std::string &msg)
{
    g_err = msg;
    return KP_ERR;
}

// the caller's workspace was too small for the result: retry with a larger `cap` (a distinct code, no message parsing)
int fail_capacity(const std::string &msg)
{
    g_err = msg;
    return KP_ERR_CAPACITY;
}

#define KP_CUDA(call)                                                                         \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail(std::string(#call) + ": " + cudaGetErrorString(e_) + " (" + __FILE__ + ":" + \
                        std::to_string(__LINE__) + ")");                                      \
    } while (0)

}  // namespace

#ifndef KP_PF_TOP
#define KP_PF_TOP 0      // prefetch the splits of the top KP_PF_TOP high positions only (0: all)
#endif
#ifndef KP_EVICT_TOP
#define KP_EVICT_TOP 0   // top high positions whose child tiles are loaded with an L2 evict-first policy (KP_EVICT_TOP in the environment)
#endif

struct kp_plan {
    KpHostPlan host;
    int device = 0;
    int sm_count = 0;
    KpTables *d_tab = nullptr;
    uint8_t *d_rowtab = nullptr;
    uint32_t *d_tiles = nullptr;
    uint8_t *d_genmask = nullptr;
    int *d_err = nullptr;
    uint32_t *d_counters = nullptr;  // one tile counter per wave, then (single-launch mode) 64 finished-tile counters
    uint8_t *d_tile_wave = nullptr;  // single-launch mode: wave of every entry of d_tiles
    uint8_t *d_tile_done = nullptr;  // single-launch mode: per-tile completion flags
    unsigned char *d_scratch = nullptr;  // staging for the small host<->device exchanges (grown on demand)
    size_t scratch_cap = 0;
    uint64_t launches = 0;
    int nwarps[2] = {0, 0};  // warps (= tiles in flight) per CTA of the DP kernel [wide]
    size_t smem_optin = 0;
    bool coop_launch = false;        // the device supports cooperative launches (backtrack: all depths in one launch)
    // tuning knobs, read from the environment ONCE, when the plan is created (tools/ab_env.py makes a plan per setting)
    // fiber kernel (kp_fiber.cuh): tables and the fiber list, when the general pattern has the shape for it
    KpFiberTables *d_ftab = nullptr;
    uint8_t *d_fiberblob = nullptr;
    uint32_t *d_fibers = nullptr;
    size_t fiber_smem[2] = {0, 0};
    int fiber_dbg = 0;               // KP_FIBER_DBG: timing experiments (results are wrong when set)
    bool use_fiber = false;          // KP_DP_KERNEL=fiber|rows: which kernel family runs the unsharded DP
    int pf_dist = KP_PF_DIST;        // KP_PF_DIST: L2 prefetch distance of the child-tile stream
    int evict_top = KP_EVICT_TOP;    // KP_EVICT_TOP: top high positions whose child tiles are loaded L2-evict-first
    bool coop_tail = true;           // KP_NO_COOP_TAIL: waves of at most one tile per SM run one CTA per tile (all warps stream)
    int pf_bulk = 0;                 // KP_PF_BULK=1: L2 prefetch by bulk copies (UBLKPF) instead of one line per lane
    int pf_top = KP_PF_TOP;          // KP_PF_TOP: only the splits of this many top high positions are prefetched (0: all)
    bool one_launch = false;         // KP_ONE_LAUNCH=1: all waves in one launch (DESIGN.md section 4)
};

// the all-N tile shape (register radix 15, two N row positions: 225 rows) gets its row pitch at compile time
#define KP_RP_NN 232
#ifndef KP_FIBER_DEFAULT
#define KP_FIBER_DEFAULT false   // which kernel family runs the unsharded DP when KP_DP_KERNEL is not set
#endif

template <bool WIDE>
static const void *dp_kernel_for_radix(int r0, int rp)
{
    switch (r0) {
    case 1: return (const void *)kp_dp_rows_kernel<1, WIDE, 0, 0>;
    case 3: return (const void *)kp_dp_rows_kernel<3, WIDE, 0, 0>;
    case 7: return (const void *)kp_dp_rows_kernel<7, WIDE, 0, 0>;
    default:
        return rp == KP_RP_NN ? (const void *)kp_dp_rows_kernel<15, WIDE, KP_RP_NN, 0>
                              : (const void *)kp_dp_rows_kernel<15, WIDE, 0, 0>;
    }
}

template <int R0, int RP, int SHARD>
static void launch_dp_r0(bool wide, int grid, int threads, size_t smem, cudaStream_t st, const KpDpParams &prm)
{
    if (wide) kp_dp_rows_kernel<R0, true, RP, SHARD><<<grid, threads, smem, st>>>(prm);
    else kp_dp_rows_kernel<R0, false, RP, SHARD><<<grid, threads, smem, st>>>(prm);
}

// the sharded DP exists for the register radix 15 only (a pattern without an N position is far too small to shard)
template <bool WIDE, int SHARD>
static const void *dp_kernel_sharded(int rp)
{
    return rp == KP_RP_NN ? (const void *)kp_dp_rows_kernel<15, WIDE, KP_RP_NN, SHARD>
                          : (const void *)kp_dp_rows_kernel<15, WIDE, 0, SHARD>;
}

// a view of one unsharded table
static KpView single_view(const kp_plan *p, const float *best, const uint16_t *flags);

// float32 sum of the leaves' held-out losses in the order of the partition tree (keys sorted ascending;
// bit 63-depth of a key tells the side taken at that depth)
static float tree_sum(const unsigned long long *keys, const float *vals, size_t lo, size_t hi, int depth)
{
    if (hi - lo == 1) return vals[lo];
    const unsigned long long bit = 1ULL << (63 - depth);
    size_t a = lo, b = hi;  // first index whose key has the bit set
    while (a < b) {
        size_t mid = (a + b) / 2;
        if (keys[mid] & bit) b = mid; else a = mid + 1;
    }
    if (a == lo || a == hi) return tree_sum(keys, vals, lo, hi, depth + 1);  // cannot happen for a well-formed tree
    volatile float l = tree_sum(keys, vals, lo, a, depth + 1), r = tree_sum(keys, vals, a, hi, depth + 1);
    volatile float sum = l + r;   // float32 add, like the reference's test_score_mem row sums
    return sum;
}

static KpView single_view(const kp_plan *p, const float *best, const uint16_t *flags)
{
    KpView v;
    memset(&v, 0, sizeof v);
    v.best[0] = best;
    v.flags[0] = flags;
    v.hw_top = (uint32_t)p->host.t.ntiles;   // tile / hw_top == 0 for every tile
    return v;
}

extern "C" {

const char *kp_last_error(void) { return g_err.c_str(); }
int kp_version(void) { return 100; }

static const void *dp_kernel_ptr(int r0, int rp, bool wide)
{
    return wide ? dp_kernel_for_radix<true>(r0, rp) : dp_kernel_for_radix<false>(r0, rp);
}

static int plan_create(const char *gen_pat, int device, bool lattice, kp_plan **out);

int kp_plan_create(const char *gen_pat, int device, kp_plan **out) { return plan_create(gen_pat, device, true, out); }

int kp_plan_create_lite(const char *gen_pat, int device, kp_plan **out) { return plan_create(gen_pat, device, false, out); }

static int plan_create(const char *gen_pat, int device, bool lattice, kp_plan **out)
{
    if (!gen_pat || !out) return fail("kp_plan_create: null argument");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(std::string("kp_plan_create: no CUDA device (") + cudaGetErrorString(e) + "); there is no CPU path");
    if (device < 0 || device >= ndev) return fail("kp_plan_create: bad device ordinal");
    KP_CUDA(cudaSetDevice(device));
    kp_plan *p = new kp_plan();
    std::string err;
    if (kp_build_host_plan(gen_pat, p->host, err, lattice)) { delete p; return fail("kp_plan_create: " + err); }
    p->device = device;
    cudaDeviceProp prop;
    KP_CUDA(cudaGetDeviceProperties(&prop, device));
    p->sm_count = prop.multiProcessorCount;
    const KpTables &t = p->host.t;
    KP_CUDA(cudaMalloc(&p->d_tab, sizeof(KpTables)));
    KP_CUDA(cudaMemcpy(p->d_tab, &t, sizeof(KpTables), cudaMemcpyHostToDevice));
    KP_CUDA(cudaMalloc(&p->d_rowtab, p->host.rowtab.size()));
    KP_CUDA(cudaMemcpy(p->d_rowtab, p->host.rowtab.data(), p->host.rowtab.size(), cudaMemcpyHostToDevice));
    KP_CUDA(cudaMalloc(&p->d_tiles, sizeof(uint32_t) * (p->host.tile_order.size() + 1)));
    KP_CUDA(cudaMemcpy(p->d_tiles, p->host.tile_order.data(), sizeof(uint32_t) * p->host.tile_order.size(), cudaMemcpyHostToDevice));
    KP_CUDA(cudaMalloc(&p->d_genmask, KP_MAXK));
    KP_CUDA(cudaMemcpy(p->d_genmask, p->host.gen_mask, KP_MAXK, cudaMemcpyHostToDevice));
    KP_CUDA(cudaMalloc(&p->d_err, sizeof(int)));
    KP_CUDA(cudaMemset(p->d_err, 0, sizeof(int)));
    KP_CUDA(cudaMalloc(&p->d_counters, sizeof(uint32_t) * 128));
    if (t.r0 == 15 && t.nhigh > 0 && lattice) {
        std::vector<uint8_t> tw(p->host.tile_order.size());
        for (size_t l = 0; l + 1 < p->host.hl_off.size(); l++)
            for (uint64_t i = p->host.hl_off[l]; i < p->host.hl_off[l + 1]; i++) tw[i] = (uint8_t)l;
        KP_CUDA(cudaMalloc(&p->d_tile_wave, tw.size()));
        KP_CUDA(cudaMemcpy(p->d_tile_wave, tw.data(), tw.size(), cudaMemcpyHostToDevice));
        KP_CUDA(cudaMalloc(&p->d_tile_done, tw.size()));
    }
    p->smem_optin = prop.sharedMemPerBlockOptin;
    if (p->host.ft.ok) {
        const KpFiberTables &f = p->host.ft;
        KP_CUDA(cudaMalloc(&p->d_ftab, sizeof(KpFiberTables)));
        KP_CUDA(cudaMemcpy(p->d_ftab, &f, sizeof(KpFiberTables), cudaMemcpyHostToDevice));
        KP_CUDA(cudaMalloc(&p->d_fiberblob, p->host.fibertab.size()));
        KP_CUDA(cudaMemcpy(p->d_fiberblob, p->host.fibertab.data(), p->host.fibertab.size(), cudaMemcpyHostToDevice));
        KP_CUDA(cudaMalloc(&p->d_fibers, sizeof(uint32_t) * (p->host.fiber_order.size() + 1)));
        KP_CUDA(cudaMemcpy(p->d_fibers, p->host.fiber_order.data(), sizeof(uint32_t) * p->host.fiber_order.size(), cudaMemcpyHostToDevice));
        for (int wide = 0; wide < 2; wide++) {
            const size_t need = kp_fiber_smem(f.ft_bytes, f.maxhs, t.tile_kmers, wide != 0).total;
            p->fiber_smem[wide] = need <= p->smem_optin ? need : 0;
        }
        KP_CUDA(cudaFuncSetAttribute((const void *)kp_dp_fiber_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)prop.sharedMemPerBlockOptin));
        KP_CUDA(cudaFuncSetAttribute((const void *)kp_dp_fiber_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)prop.sharedMemPerBlockOptin));
        p->use_fiber = KP_FIBER_DEFAULT;
        if (const char *e = getenv("KP_DP_KERNEL")) p->use_fiber = strcmp(e, "fiber") == 0;
        if (const char *e = getenv("KP_FIBER_DBG")) p->fiber_dbg = atoi(e);
    }
    p->coop_launch = prop.cooperativeLaunch != 0 && !getenv("KP_NO_COOP_BACKTRACK");
    if (const char *e = getenv("KP_PF_DIST")) p->pf_dist = atoi(e);
    if (const char *e = getenv("KP_EVICT_TOP")) p->evict_top = atoi(e);
    if (const char *e = getenv("KP_PF_TOP")) p->pf_top = atoi(e);
    if (const char *e = getenv("KP_PF_BULK")) p->pf_bulk = atoi(e);
    if (getenv("KP_NO_COOP_TAIL")) p->coop_tail = false;
    if (const char *e = getenv("KP_ONE_LAUNCH")) p->one_launch = e[0] == '1';
    for (int wide = 0; wide < 2; wide++) {
        size_t fixed = 2048 + t.rt_bytes, per_warp = t.warp_smem_bytes[wide];
        int nw = fixed < p->smem_optin ? (int)((p->smem_optin - fixed) / per_warp) : 0;
        if (nw > KP_MAX_WARPS) nw = KP_MAX_WARPS;
        p->nwarps[wide] = nw;
        // the attribute is per function, not per plan: always raise it to the device maximum
        KP_CUDA(cudaFuncSetAttribute(dp_kernel_ptr(t.r0, t.rp, wide), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)prop.sharedMemPerBlockOptin));
        if (t.r0 == 15)
            KP_CUDA(cudaFuncSetAttribute(wide ? dp_kernel_sharded<true, 3>(t.rp) : dp_kernel_sharded<false, 3>(t.rp),
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)prop.sharedMemPerBlockOptin));
    }
    *out = p;
    return 0;
}

int kp_plan_destroy(kp_plan *p)
{
    if (!p) return 0;
    cudaSetDevice(p->device);
    cudaFree(p->d_tab);
    cudaFree(p->d_rowtab);
    cudaFree(p->d_tiles);
    cudaFree(p->d_genmask);
    cudaFree(p->d_err);
    cudaFree(p->d_counters);
    cudaFree(p->d_tile_wave);
    cudaFree(p->d_tile_done);
    cudaFree(p->d_ftab);
    cudaFree(p->d_fiberblob);
    cudaFree(p->d_fibers);
    cudaFree(p->d_scratch);
    delete p;
    return 0;
}

uint64_t kp_backtrack_ws_bytes(uint64_t cap) { return (3 * cap) * sizeof(KpBtNode) + cap * (8 + 8 + 4) + 80 * 8 + 64; }

int kp_plan_get_info(const kp_plan *p, kp_plan_info *o)
{
    if (!p || !o) return fail("kp_plan_get_info: null argument");
    const KpTables &t = p->host.t;
    memset(o, 0, sizeof *o);
    o->npat = p->host.npat;
    o->nkmer = p->host.nkmer;
    o->ntiles = t.ntiles;
    o->table_elems = (uint64_t)t.ntiles * t.tile_stride;
    o->kept_elems = (uint64_t)t.ntiles * (uint64_t)t.rp;
    o->expanded_elems = (uint64_t)t.ntiles * t.tile_kmers;
    o->backtrack_ws_bytes = kp_backtrack_ws_bytes(65536);
    o->k = (uint32_t)p->host.k;
    o->nlevels = t.total_level + 1;
    o->tile_cells = t.tile_cells;
    o->tile_stride = t.tile_stride;
    o->tile_kmers = t.tile_kmers;
    o->low_positions = (uint32_t)t.nlow;
    o->register_radix = (uint32_t)t.r0;
    o->rows = (uint32_t)t.nrows;
    o->rounds = (uint32_t)t.nrounds;
    o->warps_per_cta = (uint32_t)p->nwarps[0];
    o->high_levels = (uint32_t)(p->host.hl_off.size() - 1);
    o->sm_count = (uint32_t)p->sm_count;
    return 0;
}

uint64_t kp_plan_launch_count(const kp_plan *p) { return p ? p->launches : 0; }

const char *kp_dp_kernel_name(const kp_plan *p, int wide)
{
    return p && p->use_fiber && p->fiber_smem[wide != 0] ? "kp_dp_fiber_kernel" : "kp_dp_rows_kernel";
}

int kp_pattern_offset(const kp_plan *p, uint64_t patnum, uint64_t *table_elem, uint64_t *kept_elem, uint32_t *kept_bit)
{
    if (p && !p->host.lattice) return fail("kp_pattern_offset: this plan was created without the tile lattice (kp_plan_create_lite)");
    if (!p) return fail("kp_pattern_offset: null plan");
    if (patnum >= p->host.npat) return fail("kp_pattern_offset: pattern number out of range");
    uint64_t tile; uint32_t srow, d0;
    kp_locate(p->host, patnum, &tile, &srow, &d0);
    const KpTables &t = p->host.t;
    if (table_elem) *table_elem = tile * t.tile_stride + ((uint64_t)(d0 >> 2) * t.rp + srow) * 4 + (d0 & 3);
    if (kept_elem) *kept_elem = tile * (uint64_t)t.rp + srow;
    if (kept_bit) *kept_bit = d0;
    return 0;
}

// plan-owned staging buffer: no allocator traffic on the hot host paths (stream-ordered use only)
static int scratch_reserve(kp_plan *p, size_t bytes, cudaStream_t st)
{
    if (bytes <= p->scratch_cap) return 0;
    KP_CUDA(cudaStreamSynchronize(st));
    if (p->d_scratch) KP_CUDA(cudaFree(p->d_scratch));
    p->d_scratch = nullptr;
    p->scratch_cap = 0;
    size_t cap = bytes + bytes / 2 + 4096;
    KP_CUDA(cudaMalloc(&p->d_scratch, cap));
    p->scratch_cap = cap;
    return 0;
}

static int grid_for(uint64_t n, int threads, int sm_count)
{
    uint64_t b = (n + threads - 1) / threads;
    uint64_t cap = (uint64_t)sm_count * 16;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (int)b;
}

int kp_pack_counts(kp_plan *p, const uint64_t *h_codes, const int64_t *h_pos, const int64_t *h_neg, uint64_t n,
                   int64_t *d_kmerM, int64_t *d_kmerU, void *stream)
{
    if (!p) return fail("kp_pack_counts: null plan");
    if (p->host.k > 16) return fail("kp_pack_counts: packed codes hold at most 16 positions");
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    KP_CUDA(cudaMemsetAsync(d_kmerM, 0, p->host.nkmer * 8, st));
    KP_CUDA(cudaMemsetAsync(d_kmerU, 0, p->host.nkmer * 8, st));
    if (n == 0) return 0;
    if (scratch_reserve(p, n * 24, st)) return 1;
    unsigned long long *d_codes = (unsigned long long *)p->d_scratch;
    long long *d_pos = (long long *)(d_codes + n), *d_neg = d_pos + n;
    KP_CUDA(cudaMemcpyAsync(d_codes, h_codes, n * 8, cudaMemcpyHostToDevice, st));
    KP_CUDA(cudaMemcpyAsync(d_pos, h_pos, n * 8, cudaMemcpyHostToDevice, st));
    KP_CUDA(cudaMemcpyAsync(d_neg, h_neg, n * 8, cudaMemcpyHostToDevice, st));
    KP_CUDA(cudaMemsetAsync(p->d_err, 0, sizeof(int), st));
    kp_pack_kernel<<<grid_for(n, 256, p->sm_count), 256, 0, st>>>(p->d_tab, p->d_genmask, p->host.k, d_codes, d_pos, d_neg, n,
                                                                  (long long *)d_kmerM, (long long *)d_kmerU, p->d_err);
    p->launches++;
    KP_CUDA(cudaGetLastError());
    int herr = 0;
    KP_CUDA(cudaMemcpyAsync(&herr, p->d_err, sizeof(int), cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    if (herr) return fail("kp_pack_counts: a k-mer code is not one-hot or lies outside the general pattern");
    return 0;
}

int kp_expand_counts(kp_plan *p, const int64_t *d_kmerM, const int64_t *d_kmerU, int64_t *d_expM, int64_t *d_expU,
                     void *stream)
{
    if (!p) return fail("kp_expand_counts: null plan");
    if (!p->host.lattice) return fail("kp_expand_counts: this plan was created without the tile lattice (kp_plan_create_lite)");
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    const KpTables &t = p->host.t;
    kp_expand_base_kernel<<<grid_for(p->host.nkmer, 256, p->sm_count), 256, 0, st>>>(
        p->d_tab, p->host.nkmer, (const long long *)d_kmerM, (const long long *)d_kmerU, (long long *)d_expM, (long long *)d_expU);
    p->launches++;
    for (int hi = 0; hi < t.nhigh; hi++) {
        uint64_t total = t.tile_kmers;   // elements this pass writes
        for (int h = 0; h < t.nhigh; h++) {
            const int f = t.highpos[h];
            total *= h < hi ? (uint64_t)t.radix[f] : (h == hi ? (uint64_t)(t.radix[f] - t.nbase[f]) : (uint64_t)t.nbase[f]);
        }
        if (total == 0) continue;
        kp_expand_pass_kernel<<<grid_for(total, 256, p->sm_count), 256, 0, st>>>(p->d_tab, hi, total, (long long *)d_expM,
                                                                                 (long long *)d_expU);
        p->launches++;
    }
    KP_CUDA(cudaGetLastError());
    return 0;
}

static int launch_dp(kp_plan *p, bool wide, KpDpParams prm, cudaStream_t st)
{
    if (!p->host.lattice) return fail("this plan was created without the tile lattice (kp_plan_create_lite): no DP");
    int nw = p->nwarps[wide];
    if (nw < 1) return fail("DP kernel does not fit in shared memory for this tile shape");
    size_t nhl = p->host.hl_off.size() - 1;
    const KpTables &t = p->host.t;
    if (nhl > 64) return fail("too many tile waves");
    KP_CUDA(cudaMemsetAsync(p->d_counters, 0, sizeof(uint32_t) * 128, st));
    if (p->use_fiber && p->fiber_smem[wide]) {
        // a fourth position on chip: one CTA per fiber (15 tiles), waves over the other high positions
        KpFiberParams fp;
        memset(&fp, 0, sizeof fp);
        fp.tab = p->d_tab; fp.ftab = p->d_ftab; fp.fiberblob = p->d_fiberblob;
        fp.e0 = prm.e0; fp.e1 = prm.e1; fp.s0 = prm.s0; fp.s1 = prm.s1;
        fp.alpha = prm.alpha; fp.beta = prm.beta; fp.penalty = prm.penalty;
        fp.best = prm.best; fp.flags = prm.flags;
        fp.dbg = p->fiber_dbg;
        const size_t nfl = p->host.fl_off.size() - 1;
        for (size_t l = 0; l < nfl; l++) {
            const uint64_t lo = p->host.fl_off[l], hi = p->host.fl_off[l + 1];
            if (hi == lo) continue;
            fp.fiber_list = p->d_fibers + lo;
            fp.nfibers_wave = (uint32_t)(hi - lo);
            fp.counter = p->d_counters + l;
            fp.leaf_wave = (l == 0);
            const int grid = (int)std::min<uint64_t>(hi - lo, (uint64_t)p->sm_count);
            if (wide) kp_dp_fiber_kernel<true><<<grid, KP_FIBER_THREADS, p->fiber_smem[1], st>>>(fp);
            else kp_dp_fiber_kernel<false><<<grid, KP_FIBER_THREADS, p->fiber_smem[0], st>>>(fp);
            p->launches++;
        }
        KP_CUDA(cudaGetLastError());
        return 0;
    }
    // Opt-in (KP_ONE_LAUNCH=1) for large all-N problems: ONE launch over every wave; tiles wait for their child tiles, not
    // for a kernel boundary.  Not the default: see DESIGN.md section 4.
    if (p->d_tile_done && t.ntiles >= (uint64_t)8 * p->sm_count * nw && p->one_launch) {
        KP_CUDA(cudaMemsetAsync(p->d_tile_done, 0, t.ntiles, st));
        KP_CUDA(cudaMemsetAsync(p->d_err, 0, sizeof(int), st));
        prm.tile_list = p->d_tiles;
        prm.ntiles_wave = (uint32_t)t.ntiles;
        prm.counter = p->d_counters;
        prm.leaf_wave = 0;
        prm.tile_wave = p->d_tile_wave;
        prm.tile_done = p->d_tile_done;
        prm.wave_done = p->d_counters + 64;
        prm.err = p->d_err;
        for (size_t l = 0; l < 64; l++) prm.wave_size[l] = l < nhl ? (uint32_t)(p->host.hl_off[l + 1] - p->host.hl_off[l]) : 0;
        const size_t sm = 2048 + t.rt_bytes + (size_t)nw * t.warp_smem_bytes[wide];
        if (t.rp == KP_RP_NN) launch_dp_r0<15, KP_RP_NN, 3>(wide, p->sm_count, nw * 32, sm, st, prm);
        else launch_dp_r0<15, 0, 3>(wide, p->sm_count, nw * 32, sm, st, prm);
        p->launches++;
        KP_CUDA(cudaGetLastError());
        return 0;
    }
    for (size_t l = 0; l < nhl; l++) {
        uint64_t lo = p->host.hl_off[l], hi = p->host.hl_off[l + 1];
        if (hi == lo) continue;
        prm.tile_list = p->d_tiles + lo;
        prm.ntiles_wave = (uint32_t)(hi - lo);
        prm.counter = p->d_counters + l;
        prm.leaf_wave = (l == 0);
        uint64_t ntile = hi - lo;
        const int nchunk = (t.nrows + 31) / 32;
        if (p->coop_tail && t.r0 == 15 && ntile <= (uint64_t)p->sm_count && nchunk <= KP_MAX_WARPS) {
            // at most one tile per SM (the last waves of a big lattice, every wave of a small one): a CTA per tile, every
            // warp streams one 32-row chunk of it, warp 0 runs the rounds - the wave costs a fraction of a tile latency
            const size_t smc = 2048 + t.rt_bytes + (size_t)t.warp_smem_bytes[wide];
            if (t.rp == KP_RP_NN) launch_dp_r0<15, KP_RP_NN, 4>(wide, (int)ntile, nchunk * 32, smc, st, prm);
            else launch_dp_r0<15, 0, 4>(wide, (int)ntile, nchunk * 32, smc, st, prm);
            p->launches++;
            continue;
        }
        int warps = nw;
        if (ntile < (uint64_t)p->sm_count * nw) {  // small wave: spread the tiles over all SMs
            warps = (int)((ntile + p->sm_count - 1) / p->sm_count);
            if (warps < 1) warps = 1;
        }
        uint64_t grid = (ntile + warps - 1) / warps;
        if (grid > (uint64_t)p->sm_count) grid = p->sm_count;
        size_t sm = 2048 + t.rt_bytes + (size_t)warps * t.warp_smem_bytes[wide];
        switch (t.r0) {
        case 1: launch_dp_r0<1, 0, 0>(wide, (int)grid, warps * 32, sm, st, prm); break;
        case 3: launch_dp_r0<3, 0, 0>(wide, (int)grid, warps * 32, sm, st, prm); break;
        case 7: launch_dp_r0<7, 0, 0>(wide, (int)grid, warps * 32, sm, st, prm); break;
        default:
            if (t.rp == KP_RP_NN) launch_dp_r0<15, KP_RP_NN, 0>(wide, (int)grid, warps * 32, sm, st, prm);
            else launch_dp_r0<15, 0, 0>(wide, (int)grid, warps * 32, sm, st, prm);
            break;
        }
        p->launches++;
    }
    KP_CUDA(cudaGetLastError());
    return 0;
}

static int dp_counts(kp_plan *p, const int64_t *d_expM, const int64_t *d_expU, const int64_t *d_subM, const int64_t *d_subU,
                     uint64_t max_count, double alpha, double beta, double penalty, float *d_best, uint16_t *d_kept, void *stream);

int kp_dp_single(kp_plan *p, const int64_t *d_expM, const int64_t *d_expU, uint64_t max_count, double alpha, double beta,
                 double penalty, float *d_best, uint16_t *d_kept, void *stream)
{
    return dp_counts(p, d_expM, d_expU, nullptr, nullptr, max_count, alpha, beta, penalty, d_best, d_kept, stream);
}

// the DP on the counts d_expM - d_subM, d_expU - d_subU (d_sub*: null for none)
static int dp_counts(kp_plan *p, const int64_t *d_expM, const int64_t *d_expU, const int64_t *d_subM, const int64_t *d_subU,
                     uint64_t max_count, double alpha, double beta, double penalty, float *d_best, uint16_t *d_kept, void *stream)
{
    if (!p) return fail("kp_dp_single: null plan");
    KP_CUDA(cudaSetDevice(p->device));
    bool wide = max_count > 0xFFFFFFFFull;
    KpDpParams prm;
    memset(&prm, 0, sizeof prm);
    prm.tab = p->d_tab;
    prm.rowtab = p->d_rowtab;
    prm.e0 = (const long long *)d_expM;
    prm.e1 = (const long long *)d_expU;
    prm.s0 = (const long long *)d_subM;
    prm.s1 = (const long long *)d_subU;
    prm.alpha = alpha; prm.beta = beta; prm.penalty = penalty;
    prm.best = d_best;
    prm.flags = d_kept;
    prm.pf_dist = p->pf_dist;
    prm.evict_top = p->evict_top < p->host.t.nhigh ? p->evict_top : 0;
    prm.pf_top = p->pf_top;
    prm.pf_bulk = p->pf_bulk;
    return launch_dp(p, wide, prm, (cudaStream_t)stream);
}

// breadth-first backtrack from `root`; leaves end up sorted by path key in the workspace
static int backtrack_device(kp_plan *p, const KpView &vw, void *d_ws, uint64_t cap, uint64_t root,
                            cudaStream_t st, unsigned long long **sorted_out, unsigned long long **keys_out, float **vals_out,
                            unsigned long long **ctr_out)
{
    KpBtNode *fa = (KpBtNode *)d_ws, *fb = fa + cap, *leaves = fb + cap;
    unsigned long long *sorted = (unsigned long long *)(leaves + cap);
    unsigned long long *keys = sorted + cap;
    unsigned long long *ctr = keys + cap;   // [0] leaves, [1] overflow, [2 + d] nodes at depth d
    float *vals = (float *)(ctr + 80);
    kp_backtrack_init_kernel<<<1, 128, 0, st>>>(fa, root, ctr);
    const int levels = (int)p->host.t.total_level + 1;
    int grid = (int)((cap + 7) / 8);
    if (grid > p->sm_count * 2) grid = p->sm_count * 2;
    // all depths in one cooperative launch (grid-wide barrier between depths); one launch per depth if the device
    // cannot run the grid co-resident
    bool fused = false;
    if (p->coop_launch) {
        int nlev = levels < 64 ? levels : 64;
        int cgrid = grid < p->sm_count ? grid : p->sm_count;
        const KpTables *a_tab = p->d_tab;
        const uint8_t *a_row = p->d_rowtab;
        void *args[] = {(void *)&a_tab, (void *)&a_row, (void *)&vw, (void *)&nlev, (void *)&fa, (void *)&fb, (void *)&leaves,
                        (void *)&cap, (void *)&ctr};
        if (cudaLaunchCooperativeKernel((const void *)kp_backtrack_all_kernel, dim3(cgrid), dim3(256), args, 0, st) == cudaSuccess) {
            fused = true;
            p->launches++;
        } else {
            cudaGetLastError();
        }
    }
    for (int d = 0; !fused && d < levels && d < 64; d++) {
        kp_backtrack_level_kernel<<<grid, 256, 0, st>>>(p->d_tab, p->d_rowtab, vw, d, (d & 1) ? fb : fa,
                                                        (d & 1) ? fa : fb, leaves, cap, ctr);
        p->launches++;
    }
    kp_backtrack_sort_kernel<<<p->sm_count, 256, 0, st>>>(leaves, ctr, cap, sorted, keys);
    p->launches += 2;
    KP_CUDA(cudaGetLastError());
    *sorted_out = sorted; *keys_out = keys; *vals_out = vals; *ctr_out = ctr;
    return 0;
}

int kp_backtrack(kp_plan *p, const float *d_best, const uint16_t *d_kept, void *d_ws, uint64_t cap, uint64_t root,
                 uint64_t *h_patnums, uint64_t *n_out, void *stream)
{
    if (!p || !d_ws || !h_patnums || !n_out) return fail("kp_backtrack: null argument");
    if (p->host.t.total_level > 64) return fail("kp_backtrack: more than 64 levels");
    if (root == UINT64_MAX) root = p->host.npat - 1;
    if (root >= p->host.npat) return fail("kp_backtrack: root out of range");
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    unsigned long long *sorted, *keys, *ctr;
    float *vals;
    if (backtrack_device(p, single_view(p, d_best, d_kept), d_ws, cap, root, st, &sorted, &keys, &vals, &ctr)) return 1;
    unsigned long long hc[2] = {0, 0};
    int herr = 0;
    KP_CUDA(cudaMemcpyAsync(hc, ctr, sizeof hc, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaMemcpyAsync(&herr, p->d_err, sizeof herr, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    if (herr == 2) return fail("kp_backtrack: the DP gave up waiting for a child tile (internal error)");
    *n_out = hc[0];
    if (hc[1] || hc[0] > cap) return fail_capacity("kp_backtrack: partition larger than the workspace capacity");
    KP_CUDA(cudaMemcpyAsync(h_patnums, sorted, hc[0] * 8, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int kp_cv_heldout(kp_plan *p, const float *d_train, const uint16_t *d_kept, const int64_t *d_expMtot, const int64_t *d_expUtot,
                  const int64_t *d_expMtest, const int64_t *d_expUtest, double alpha, double beta_fold, double penalty,
                  uint64_t root, void *d_ws, uint64_t cap, float *h_test, void *stream)
{
    if (!p || !d_ws || !h_test) return fail("kp_cv_heldout: null argument");
    if (root == UINT64_MAX) root = p->host.npat - 1;
    if (root >= p->host.npat) return fail("kp_cv_heldout: root out of range");
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    unsigned long long *sorted, *keys, *ctr;
    float *vals;
    if (backtrack_device(p, single_view(p, d_train, d_kept), d_ws, cap, root, st, &sorted, &keys, &vals, &ctr)) return 1;
    kp_cv_leaf_kernel<<<p->sm_count, 128, 0, st>>>(p->d_tab, p->d_rowtab, (const long long *)d_expMtot, (const long long *)d_expUtot,
                                                   (const long long *)d_expMtest, (const long long *)d_expUtest, alpha, beta_fold,
                                                   penalty, sorted, ctr, cap, vals);
    p->launches++;
    KP_CUDA(cudaGetLastError());
    unsigned long long hc[2] = {0, 0};
    KP_CUDA(cudaMemcpyAsync(hc, ctr, sizeof hc, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    if (hc[1] || hc[0] > cap) return fail_capacity("kp_cv_heldout: partition larger than the workspace capacity");
    if (hc[0] == 0) return fail("kp_cv_heldout: the backtrack produced no leaf (internal error)");
    std::vector<unsigned long long> hk(hc[0]);
    std::vector<float> hv(hc[0]);
    KP_CUDA(cudaMemcpyAsync(hk.data(), keys, hc[0] * 8, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaMemcpyAsync(hv.data(), vals, hc[0] * 4, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    *h_test = tree_sum(hk.data(), hv.data(), 0, hc[0], 0);
    return 0;
}

int kp_dp_cv_job(kp_plan *p, const int64_t *d_expMtot, const int64_t *d_expUtot, const int64_t *d_expMtest,
                 const int64_t *d_expUtest, uint64_t max_count, double alpha, double beta_fold, double penalty,
                 float *d_train, uint16_t *d_kept, void *d_ws, uint64_t cap, float *h_top, void *stream)
{
    if (!p || !d_expMtest || !d_expUtest) return fail("kp_dp_cv_job: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    const KpTables &t = p->host.t;
    // train counts = total - held-out: the subtraction commutes with the sums of the expansion, so it is done by the DP
    // kernel (and the leaf kernel) when they read the tile's base counts; no train table is materialised
    if (dp_counts(p, d_expMtot, d_expUtot, d_expMtest, d_expUtest, max_count, alpha, beta_fold, penalty, d_train, d_kept, stream))
        return 1;
    if (h_top) {
        if (int rc = kp_cv_heldout(p, d_train, d_kept, d_expMtot, d_expUtot, d_expMtest, d_expUtest, alpha, beta_fold, penalty,
                                   UINT64_MAX, d_ws, cap, h_top + 1, stream))
            return rc;
        uint64_t tile; uint32_t srow, d0;
        kp_locate(p->host, p->host.npat - 1, &tile, &srow, &d0);
        size_t top = (size_t)tile * t.tile_stride + ((size_t)(d0 >> 2) * t.rp + srow) * 4 + (d0 & 3);
        KP_CUDA(cudaMemcpyAsync(h_top, d_train + top, sizeof(float), cudaMemcpyDeviceToHost, st));
        KP_CUDA(cudaStreamSynchronize(st));
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// A CV job without a host round trip: kp_cv_job_enqueue queues the DP, the backtrack, the leaf kernel and the copies of
// their results into a (pinned) host staging area and returns at once; kp_cv_job_finish, called after the stream has
// passed that point (an event the caller records), does the host part (the float32 tree sum).  With two train tables
// in rotation the next job's DP is queued before the previous job's results are read, so the GPU never waits for the host.
// Staging layout: u64 leaves, u64 overflow, f32 train loss of the general pattern, pad to 32 bytes; u64 keys[cap]; f32 vals[cap].
// ---------------------------------------------------------------------------------------------------
uint64_t kp_cv_stage_bytes(uint64_t cap) { return 32 + cap * 12; }

int kp_cv_job_enqueue(kp_plan *p, const int64_t *d_expMtot, const int64_t *d_expUtot, const int64_t *d_expMtest,
                      const int64_t *d_expUtest, uint64_t max_count, double alpha, double beta_fold, double penalty,
                      float *d_train, uint16_t *d_kept, void *d_ws, uint64_t cap, void *h_stage, void *stream)
{
    if (!p || !d_expMtest || !d_expUtest || !d_ws || !h_stage) return fail("kp_cv_job_enqueue: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    const KpTables &t = p->host.t;
    if (dp_counts(p, d_expMtot, d_expUtot, d_expMtest, d_expUtest, max_count, alpha, beta_fold, penalty, d_train, d_kept, stream))
        return 1;
    unsigned long long *sorted, *keys, *ctr;
    float *vals;
    if (backtrack_device(p, single_view(p, d_train, d_kept), d_ws, cap, p->host.npat - 1, st, &sorted, &keys, &vals, &ctr)) return 1;
    kp_cv_leaf_kernel<<<p->sm_count, 128, 0, st>>>(p->d_tab, p->d_rowtab, (const long long *)d_expMtot, (const long long *)d_expUtot,
                                                   (const long long *)d_expMtest, (const long long *)d_expUtest, alpha, beta_fold,
                                                   penalty, sorted, ctr, cap, vals);
    p->launches++;
    KP_CUDA(cudaGetLastError());
    unsigned char *h = (unsigned char *)h_stage;
    uint64_t tile; uint32_t srow, d0;
    kp_locate(p->host, p->host.npat - 1, &tile, &srow, &d0);
    const size_t top = (size_t)tile * t.tile_stride + ((size_t)(d0 >> 2) * t.rp + srow) * 4 + (d0 & 3);
    KP_CUDA(cudaMemcpyAsync(h, ctr, 16, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaMemcpyAsync(h + 16, d_train + top, sizeof(float), cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaMemcpyAsync(h + 32, keys, cap * 8, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaMemcpyAsync(h + 32 + cap * 8, vals, cap * 4, cudaMemcpyDeviceToHost, st));
    return 0;
}

int kp_cv_job_finish(const void *h_stage, uint64_t cap, float *h_top)
{
    if (!h_stage || !h_top) return fail("kp_cv_job_finish: null argument");
    const unsigned char *h = (const unsigned char *)h_stage;
    unsigned long long hc[2];
    memcpy(hc, h, 16);
    if (hc[1] || hc[0] > cap) return fail_capacity("kp_cv_job_finish: partition larger than the workspace capacity");
    if (hc[0] == 0) return fail("kp_cv_job_finish: the backtrack produced no leaf (internal error)");
    memcpy(h_top, h + 16, sizeof(float));
    h_top[1] = tree_sum((const unsigned long long *)(h + 32), (const float *)(h + 32 + cap * 8), 0, hc[0], 0);
    return 0;
}

int kp_split_codes(kp_plan *p, const float *d_best, const uint16_t *d_kept, const uint64_t *h_patnums, uint64_t n,
                   uint8_t *h_codes, void *stream)
{
    if (!p) return fail("kp_split_codes: null plan");
    if (n == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    if (scratch_reserve(p, n * 9, st)) return 1;
    unsigned long long *d_pat = (unsigned long long *)p->d_scratch;
    uint8_t *d_codes = (uint8_t *)(d_pat + n);
    KP_CUDA(cudaMemcpyAsync(d_pat, h_patnums, n * 8, cudaMemcpyHostToDevice, st));
    kp_split_codes_kernel<<<grid_for(n, 256, p->sm_count), 256, 0, st>>>(p->d_tab, p->d_rowtab, single_view(p, d_best, d_kept), d_pat, n, d_codes);
    p->launches++;
    KP_CUDA(cudaGetLastError());
    KP_CUDA(cudaMemcpyAsync(h_codes, d_codes, n, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int kp_gather_table(kp_plan *p, const float *d_table, uint64_t first, uint64_t n, float *h_out, void *stream)
{
    if (!p) return fail("kp_gather_table: null plan");
    if (n == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    if (scratch_reserve(p, n * 4, st)) return 1;
    float *d_out = (float *)p->d_scratch;
    kp_gather_kernel<<<grid_for(n, 256, p->sm_count), 256, 0, st>>>(p->d_tab, p->d_rowtab, single_view(p, d_table, nullptr), nullptr, first, n, d_out);
    p->launches++;
    KP_CUDA(cudaGetLastError());
    KP_CUDA(cudaMemcpyAsync(h_out, d_out, n * 4, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int kp_gather_kept(kp_plan *p, const uint16_t *d_kept, uint64_t first, uint64_t n, uint8_t *h_out, void *stream)
{
    if (!p) return fail("kp_gather_kept: null plan");
    if (n == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    if (scratch_reserve(p, n, st)) return 1;
    uint8_t *d_out = (uint8_t *)p->d_scratch;
    kp_gather_flags_kernel<<<grid_for(n, 256, p->sm_count), 256, 0, st>>>(p->d_tab, p->d_rowtab, single_view(p, nullptr, d_kept), nullptr, first, n, d_out);
    p->launches++;
    KP_CUDA(cudaGetLastError());
    KP_CUDA(cudaMemcpyAsync(h_out, d_out, n, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// scores / kept-whole flags / split codes of arbitrary patterns of an unsharded table (any of the outputs may be null)
int kp_gather_patterns(kp_plan *p, const float *d_table, const uint16_t *d_kept, const uint64_t *h_patnums, uint64_t n,
                       float *h_best, uint8_t *h_kept, uint8_t *h_codes, void *stream)
{
    if (!p || !h_patnums) return fail("kp_gather_patterns: null argument");
    if (!p->host.lattice) return fail("kp_gather_patterns: this plan was created without the tile lattice (kp_plan_create_lite)");
    if ((h_best || h_codes) && !d_table) return fail("kp_gather_patterns: scores and split codes need the score table");
    if ((h_kept || h_codes) && !d_kept) return fail("kp_gather_patterns: kept flags and split codes need the kept-whole table");
    if (n == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    if (scratch_reserve(p, n * 16, st)) return 1;
    unsigned long long *d_pat = (unsigned long long *)p->d_scratch;
    float *d_val = (float *)(d_pat + n);
    uint8_t *d_k = (uint8_t *)(d_val + n), *d_c = d_k + n;
    KP_CUDA(cudaMemcpyAsync(d_pat, h_patnums, n * 8, cudaMemcpyHostToDevice, st));
    const int grid = grid_for(n, 256, p->sm_count);
    const KpView vw = single_view(p, d_table, d_kept);
    if (h_best) { kp_gather_kernel<<<grid, 256, 0, st>>>(p->d_tab, p->d_rowtab, vw, d_pat, 0, n, d_val); p->launches++; }
    if (h_kept) { kp_gather_flags_kernel<<<grid, 256, 0, st>>>(p->d_tab, p->d_rowtab, vw, d_pat, 0, n, d_k); p->launches++; }
    if (h_codes) { kp_split_codes_kernel<<<grid, 256, 0, st>>>(p->d_tab, p->d_rowtab, vw, d_pat, n, d_c); p->launches++; }
    KP_CUDA(cudaGetLastError());
    if (h_best) KP_CUDA(cudaMemcpyAsync(h_best, d_val, n * 4, cudaMemcpyDeviceToHost, st));
    if (h_kept) KP_CUDA(cudaMemcpyAsync(h_kept, d_k, n, cudaMemcpyDeviceToHost, st));
    if (h_codes) KP_CUDA(cudaMemcpyAsync(h_codes, d_c, n, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int kp_pattern_counts(kp_plan *p, const int64_t *d_kmerM, const int64_t *d_kmerU, const uint64_t *h_patnums, uint64_t n,
                      int64_t *h_M, int64_t *h_U, void *stream)
{
    if (!p) return fail("kp_pattern_counts: null plan");
    if (n == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    if (scratch_reserve(p, n * 24, st)) return 1;
    unsigned long long *d_pat = (unsigned long long *)p->d_scratch;
    long long *d_out = (long long *)(d_pat + n);
    KP_CUDA(cudaMemcpyAsync(d_pat, h_patnums, n * 8, cudaMemcpyHostToDevice, st));
    const int pc_grid = (int)std::min<uint64_t>(n, (uint64_t)p->sm_count * 16);
    kp_pattern_counts_kernel<<<pc_grid, 256, 0, st>>>(p->d_tab, n, (const long long *)d_kmerM, (const long long *)d_kmerU,
                                                      d_pat, d_out, d_out + n);
    p->launches++;
    KP_CUDA(cudaGetLastError());
    KP_CUDA(cudaMemcpyAsync(h_M, d_out, n * 8, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaMemcpyAsync(h_U, d_out + n, n * 8, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// ===================================================================================================
// Scoring a given partition.  Both entries lay out the partition in the plan's scratch: the uploaded pattern numbers,
// their packed subsets, the member offsets (n + 1) and the scan's block sums; part_prepare returns the member total.
// ===================================================================================================
struct PartLayout {
    unsigned long long *pat, *pm, *offs, *bsum;
};

static size_t part_bytes(uint64_t n) { return (3 * n + 1 + 1024) * 8; }   // the caller's own arrays follow

static PartLayout part_layout(const kp_plan *p, uint64_t n)
{
    PartLayout L;
    L.pat = (unsigned long long *)p->d_scratch;
    L.pm = L.pat + n;
    L.offs = L.pm + n;
    L.bsum = L.offs + n + 1;
    return L;
}

static int part_check(const kp_plan *p, const char *what, const uint64_t *h_patnums, uint64_t n)
{
    if (!p) return fail(std::string(what) + ": null plan");
    if (!h_patnums || n == 0) return fail(std::string(what) + ": empty partition");
    if (n >= KP_OWNER_EMPTY) return fail(std::string(what) + ": too many patterns (owners are uint32)");
    for (uint64_t i = 0; i < n; i++)
        if (h_patnums[i] >= p->host.npat) return fail(std::string(what) + ": pattern number out of range");
    return 0;
}

// after scratch_reserve: upload the patterns and scan their sizes (synchronises to read the total)
static int part_prepare(kp_plan *p, const uint64_t *h_patnums, uint64_t n, cudaStream_t st, uint64_t *total)
{
    const PartLayout L = part_layout(p, n);
    KP_CUDA(cudaMemcpyAsync(L.pat, h_patnums, n * 8, cudaMemcpyHostToDevice, st));
    const uint64_t nb = std::min<uint64_t>(1024, (n + 255) / 256), per = (n + nb - 1) / nb;
    kp_part_prep_kernel<<<(unsigned)nb, 256, 0, st>>>(p->d_tab, L.pat, n, per, L.pm, L.bsum);
    kp_part_scan_kernel<<<1, 256, 0, st>>>(L.bsum, (unsigned)nb, L.offs, n);
    kp_part_offsets_kernel<<<(unsigned)nb, 256, 0, st>>>(p->d_tab, L.pm, n, per, L.bsum, L.offs);
    p->launches += 3;
    KP_CUDA(cudaGetLastError());
    unsigned long long tot = 0;
    KP_CUDA(cudaMemcpyAsync(&tot, L.offs + n, 8, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    *total = tot;
    return 0;
}

int kp_partition_assign(kp_plan *p, const uint64_t *h_patnums, uint64_t n, uint32_t *d_owner, uint64_t *h_conflict,
                        uint64_t *h_uncovered, void *stream)
{
    if (part_check(p, "kp_partition_assign", h_patnums, n)) return KP_ERR;
    if (!d_owner || !h_conflict || !h_uncovered) return fail("kp_partition_assign: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    if (scratch_reserve(p, part_bytes(n) + 16, st)) return KP_ERR;
    const PartLayout L = part_layout(p, n);
    unsigned long long *d_res = L.bsum + 1024;
    uint64_t total = 0;
    if (part_prepare(p, h_patnums, n, st, &total)) return KP_ERR;
    const uint64_t nkmer = p->host.nkmer;
    KP_CUDA(cudaMemsetAsync(d_owner, 0xFF, nkmer * 4, st));
    KP_CUDA(cudaMemsetAsync(d_res, 0xFF, 16, st));
    const int grid = p->sm_count * 8;
    unsigned long long res[2] = {~0ull, ~0ull};
    // Chunks of nkmer members.  Past the first chunk a conflict is certain (more members than k-mers), so at most two
    // chunks run before the loop stops, however much the file over-covers.
    for (uint64_t lo = 0; lo < total; lo += nkmer) {
        const uint64_t hi = std::min<uint64_t>(total, lo + nkmer);
        kp_part_assign_kernel<<<grid, 256, 0, st>>>(p->d_tab, L.pm, L.offs, n, lo, hi, d_owner, d_res);
        p->launches++;
        KP_CUDA(cudaGetLastError());
        if (hi == total) break;
        KP_CUDA(cudaMemcpyAsync(res, d_res, 8, cudaMemcpyDeviceToHost, st));
        KP_CUDA(cudaStreamSynchronize(st));
        if (res[0] != ~0ull) break;
    }
    KP_CUDA(cudaMemcpyAsync(res, d_res, 8, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    if (res[0] == ~0ull) {   // the owner table is complete only when no chunk was cut short
        kp_part_cover_kernel<<<grid_for(nkmer, 256, p->sm_count), 256, 0, st>>>(d_owner, nkmer, d_res);
        p->launches++;
        KP_CUDA(cudaGetLastError());
        KP_CUDA(cudaMemcpyAsync(res, d_res, 16, cudaMemcpyDeviceToHost, st));
        KP_CUDA(cudaStreamSynchronize(st));
    }
    *h_conflict = res[0] == ~0ull ? 0 : res[0] + 1;
    *h_uncovered = res[0] != ~0ull || res[1] == ~0ull ? 0 : res[1] + 1;
    return 0;
}

int kp_partition_score(kp_plan *p, const uint64_t *h_patnums, const double *h_rate, uint64_t n, const int64_t *d_kmerM,
                       const int64_t *d_kmerU, const uint32_t *d_owner, double *d_kmer_rate, int64_t *h_M, int64_t *h_U,
                       double *h_t, void *stream)
{
    if (part_check(p, "kp_partition_score", h_patnums, n)) return KP_ERR;
    if (!h_rate || !d_kmerM || !d_kmerU || !h_M || !h_U || !h_t) return fail("kp_partition_score: null argument");
    if (d_kmer_rate && !d_owner) return fail("kp_partition_score: the per-k-mer rates need the owner table");
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    if (scratch_reserve(p, part_bytes(n) + 4 * n * 8, st)) return KP_ERR;
    const PartLayout L = part_layout(p, n);
    unsigned long long *d_M = (unsigned long long *)((unsigned char *)p->d_scratch + part_bytes(n)), *d_U = d_M + n;
    double *d_rate = (double *)(d_U + n), *d_t = d_rate + n;
    uint64_t total = 0;
    if (part_prepare(p, h_patnums, n, st, &total)) return KP_ERR;
    if (total > p->host.nkmer) return fail("kp_partition_score: the patterns have more members than there are k-mers (they overlap)");
    KP_CUDA(cudaMemcpyAsync(d_rate, h_rate, n * 8, cudaMemcpyHostToDevice, st));
    KP_CUDA(cudaMemsetAsync(d_M, 0, 2 * n * 8, st));
    kp_part_counts_kernel<<<p->sm_count * 8, 256, 0, st>>>(p->d_tab, L.pm, L.offs, n, total, (const long long *)d_kmerM,
                                                           (const long long *)d_kmerU, d_M, d_U);
    kp_part_terms_kernel<<<grid_for(n, 256, p->sm_count), 256, 0, st>>>(d_M, d_U, d_rate, n, d_t);
    p->launches += 2;
    if (d_kmer_rate) {
        kp_part_kmer_rate_kernel<<<grid_for(p->host.nkmer, 256, p->sm_count), 256, 0, st>>>(d_owner, d_rate, n, p->host.nkmer,
                                                                                           d_kmer_rate);
        p->launches++;
    }
    KP_CUDA(cudaGetLastError());
    KP_CUDA(cudaMemcpyAsync(h_M, d_M, n * 8, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaMemcpyAsync(h_U, d_U, n * 8, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaMemcpyAsync(h_t, d_t, n * 8, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// ===================================================================================================
// Applying a partition along sequences (DESIGN §4c).  Nothing here synchronises: the caller overlaps the next chunk's
// upload with the scan.
// ===================================================================================================
int kp_kmer_rates(kp_plan *p, const uint32_t *d_owner, const double *h_rate, uint64_t n, double *d_kmer_rate, void *stream)
{
    if (!p) return fail("kp_kmer_rates: null plan");
    if (!d_owner || !h_rate || !d_kmer_rate || n == 0) return fail("kp_kmer_rates: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    if (scratch_reserve(p, n * 8, st)) return KP_ERR;
    double *d_rate = (double *)p->d_scratch;
    KP_CUDA(cudaMemcpyAsync(d_rate, h_rate, n * 8, cudaMemcpyHostToDevice, st));
    kp_part_kmer_rate_kernel<<<grid_for(p->host.nkmer, 256, p->sm_count), 256, 0, st>>>(d_owner, d_rate, n, p->host.nkmer,
                                                                                       d_kmer_rate);
    p->launches++;
    KP_CUDA(cudaGetLastError());
    KP_CUDA(cudaStreamSynchronize(st));   // the scratch is reused by the next call
    return 0;
}

int kp_seq_scan(kp_plan *p, const uint8_t *d_seq, uint64_t seq_base, uint64_t seq_len, uint64_t rec_len, uint64_t pos0,
                uint64_t pos1, int both, const double *d_kmer_rate, const uint32_t *d_tasks, uint64_t ntask, double *d_sum,
                int64_t *d_n, float *d_track, const uint32_t *d_count_mask, int64_t *d_counts, void *stream)
{
    if (!p) return fail("kp_seq_scan: null plan");
    const int k = p->host.k, c = k / 2;
    if (!d_seq || !d_kmer_rate || !d_sum || !d_n) return fail("kp_seq_scan: null argument");
    if ((uintptr_t)d_seq & 15) return fail("kp_seq_scan: the sequence buffer must be 16-byte aligned");
    if (both && k % 2 == 0) return fail("kp_seq_scan: both strands need an odd k");
    if (pos0 % KP_SEQ_PIECE || pos0 > pos1 || pos1 > rec_len) return fail("kp_seq_scan: bad position range");
    // every window of [pos0, pos1) that lies in the record must lie in the given bytes
    const uint64_t need_lo = pos0 >= (uint64_t)c ? pos0 - c : 0, need_hi = std::min<uint64_t>(rec_len, pos1 + (k - 1 - c));
    if (pos1 > pos0 && (seq_base > need_lo || seq_base + seq_len < need_hi || seq_base + seq_len > rec_len))
        return fail("kp_seq_scan: the sequence bytes do not cover the windows of the positions");
    if (d_tasks && (d_track || d_counts)) return fail("kp_seq_scan: tracks and counts come from the whole-piece pass");
    if (pos1 == pos0 || (d_tasks && ntask == 0)) return 0;
    if (!d_tasks && (pos1 - pos0 + KP_SEQ_PIECE - 1) / KP_SEQ_PIECE > 0x7FFFFFFFull) return fail("kp_seq_scan: too many pieces");
    if (d_tasks && ntask > 0x7FFFFFFFull) return fail("kp_seq_scan: too many tasks");
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    KpSeqScan a;
    a.seq = d_seq;
    a.seq_base = seq_base;
    a.seq_len = seq_len;
    a.rec_len = rec_len;
    a.pos0 = pos0;
    a.pos1 = pos1;
    a.kmer_rate = d_kmer_rate;
    a.tasks = d_tasks;
    a.sum = d_sum;
    a.n = (unsigned long long *)d_n;
    a.track = d_track;
    a.count_mask = d_count_mask;
    a.counts = (unsigned long long *)d_counts;
    a.k = k;
    a.c = c;
    const unsigned grid = (unsigned)(d_tasks ? ntask : (pos1 - pos0 + KP_SEQ_PIECE - 1) / KP_SEQ_PIECE);
    if (both) kp_seq_scan_kernel<true><<<grid, KP_SEQ_THREADS, 0, st>>>(p->d_tab, p->d_genmask, a);
    else kp_seq_scan_kernel<false><<<grid, KP_SEQ_THREADS, 0, st>>>(p->d_tab, p->d_genmask, a);
    p->launches++;
    KP_CUDA(cudaGetLastError());
    return 0;
}

int kp_snv_counts(kp_plan *p, const uint8_t *d_seq, uint64_t seq_base, uint64_t seq_len, uint64_t rec_len, uint64_t pos0,
                  uint64_t pos1, int both, const int64_t *d_pos, const uint8_t *d_ref_alt, uint64_t n, const int *alt_slot,
                  const uint32_t *d_count_mask, int64_t *d_counts, uint8_t *d_status, void *stream)
{
    if (!p) return fail("kp_snv_counts: null plan");
    const int k = p->host.k, c = k / 2;
    if (!alt_slot) return fail("kp_snv_counts: null argument");
    for (int a = 0; a < 4; a++)
        if (alt_slot[a] < -1 || alt_slot[a] > 3) return fail("kp_snv_counts: an alt slot must be -1..3");
    if (both && k % 2 == 0) return fail("kp_snv_counts: both strands need an odd k");
    if (pos0 > pos1 || pos1 > rec_len) return fail("kp_snv_counts: bad position range");
    if (n == 0) return 0;
    if (!d_seq || !d_pos || !d_ref_alt || !d_counts || !d_status) return fail("kp_snv_counts: null argument");
    if (((uintptr_t)d_pos & 7) || ((uintptr_t)d_counts & 7)) return fail("kp_snv_counts: d_pos and d_counts must be 8-byte aligned");
    const uint64_t need_lo = pos0 >= (uint64_t)c ? pos0 - c : 0, need_hi = std::min<uint64_t>(rec_len, pos1 + (k - 1 - c));
    if (pos1 > pos0 && (seq_base > need_lo || seq_base + seq_len < need_hi || seq_base + seq_len > rec_len))
        return fail("kp_snv_counts: the sequence bytes do not cover the windows of the positions");
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    KpSnvCount a;
    a.seq = d_seq;
    a.seq_base = seq_base;
    a.seq_len = seq_len;
    a.rec_len = rec_len;
    a.pos0 = pos0;
    a.pos1 = pos1;
    a.pos = (const long long *)d_pos;
    a.ref_alt = d_ref_alt;
    a.n = n;
    a.nkmer = p->host.nkmer;
    for (int x = 0; x < 4; x++) a.alt_slot[x] = alt_slot[x];
    a.count_mask = d_count_mask;
    a.counts = (unsigned long long *)d_counts;
    a.status = d_status;
    a.k = k;
    a.c = c;
    const int grid = grid_for(n, 256, p->sm_count);
    if (both) kp_snv_count_kernel<true><<<grid, 256, 0, st>>>(p->d_tab, p->d_genmask, a);
    else kp_snv_count_kernel<false><<<grid, 256, 0, st>>>(p->d_tab, p->d_genmask, a);
    p->launches++;
    KP_CUDA(cudaGetLastError());
    return 0;
}

int kp_region_sums(kp_plan *p, const double *d_piece_sum, const int64_t *d_piece_n, const double *d_task_sum,
                   const int64_t *d_task_n, const int64_t *d_regions, uint64_t n, double *d_sum, int64_t *d_n, void *stream)
{
    if (!p) return fail("kp_region_sums: null plan");
    if (n == 0) return 0;
    if (!d_piece_sum || !d_piece_n || !d_regions || !d_sum || !d_n) return fail("kp_region_sums: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    kp_region_sum_kernel<<<grid_for(n, 256, p->sm_count), 256, 0, st>>>(
        d_piece_sum, (const unsigned long long *)d_piece_n, d_task_sum, (const unsigned long long *)d_task_n,
        (const long long *)d_regions, n, d_sum, (unsigned long long *)d_n);
    p->launches++;
    KP_CUDA(cudaGetLastError());
    return 0;
}

// ===================================================================================================
// One DP sharded over the GPUs of a node (SURVEY 8f.3).  The score table is split by the digit of the top high
// position; every rank runs the same waves on its own tiles and reads the children that live on a peer straight
// from the peer's memory (NVLink) inside the DP kernel.  The caller puts a barrier between the waves.
// ===================================================================================================
struct kp_shard {
    kp_plan *plan = nullptr;
    int rank = 0, world = 1;
    bool replicate = false;          // every rank holds a full-size table and finished tiles are pushed to their readers
    uint32_t hw_top = 0, radix_top = 0, nslots = 0;
    uint64_t local_tiles = 0;
    float *d_best = nullptr;         // this rank's shard (plain cudaMalloc, so that it can be exported over CUDA IPC)
    uint16_t *d_kept = nullptr;
    KpView view;
    uint32_t *d_tiles = nullptr;     // this rank's tiles, wave by wave (global tile numbers, ascending)
    std::vector<uint64_t> hl_off;    // wave offsets into d_tiles
    uint32_t *d_counters = nullptr;
};


// Two-dimensional shard ownership, improved by a deterministic local search (every rank runs it and gets the same table).
// A tile must be pushed to every rank that owns one of its parents along either of the two top positions, and the DP is
// NVLink-bound (DESIGN.md section 6), so the search minimises the largest inbound (and outbound) cell count of any rank
// while keeping every wave evenly spread: cells of the same level hold the same number of tiles in every wave.
// Start: owner = (i_top + i_second) mod world.  At eight ranks the busiest rank's inbound volume falls from 128 to about
// 70 of the 225 cells (one-dimensional ownership: 195).
static void optimise_cell_owners(const KpTables &t, int e1, int e2, int world, std::vector<uint8_t> &owner)
{
    const int r1 = t.radix[e1], r2 = t.radix[e2], ncell = r1 * r2;
    auto pc = [](unsigned m) { return (int)((m & 1) + ((m >> 1) & 1) + ((m >> 2) & 1) + ((m >> 3) & 1)); };
    std::vector<std::vector<int>> sup1(r1), sup2(r2);
    for (int d = 0; d < r1; d++)
        for (int q = 0; q < r1; q++)
            if (q != d && (t.digit_mask[e1][d] & t.digit_mask[e1][q]) == t.digit_mask[e1][d]) sup1[d].push_back(q);
    for (int d = 0; d < r2; d++)
        for (int q = 0; q < r2; q++)
            if (q != d && (t.digit_mask[e2][d] & t.digit_mask[e2][q]) == t.digit_mask[e2][d]) sup2[d].push_back(q);
    std::vector<int> lvl(ncell);
    int nlvl = 0;
    for (int d1 = 0; d1 < r1; d1++)
        for (int d2 = 0; d2 < r2; d2++) {
            lvl[d2 + r2 * d1] = pc(t.digit_mask[e1][d1]) + pc(t.digit_mask[e2][d2]) - 2;
            nlvl = std::max(nlvl, lvl[d2 + r2 * d1] + 1);
        }
    std::vector<int> inb(world), outb(world), wl((size_t)nlvl * world);
    auto cost = [&]() {
        std::fill(inb.begin(), inb.end(), 0);
        std::fill(outb.begin(), outb.end(), 0);
        std::fill(wl.begin(), wl.end(), 0);
        for (int d1 = 0; d1 < r1; d1++)
            for (int d2 = 0; d2 < r2; d2++) {
                const int c = d2 + r2 * d1, o = owner[c];
                wl[(size_t)lvl[c] * world + o]++;
                unsigned dest = 0;
                for (int q : sup1[d1]) dest |= 1u << owner[d2 + r2 * q];
                for (int q : sup2[d2]) dest |= 1u << owner[q + r2 * d1];
                dest &= ~(1u << o);
                for (int r = 0; r < world; r++)
                    if ((dest >> r) & 1u) { inb[r]++; outb[o]++; }
            }
        double imb = 0;
        std::vector<int> own(world, 0);
        for (int l = 0; l < nlvl; l++) {
            int mx = 0, sum = 0;
            for (int r = 0; r < world; r++) {
                mx = std::max(mx, wl[(size_t)l * world + r]);
                sum += wl[(size_t)l * world + r];
                own[r] += wl[(size_t)l * world + r];
            }
            imb += mx - (double)sum / world;
        }
        imb += *std::max_element(own.begin(), own.end()) - (double)ncell / world;   // and the whole table evenly, too
        return *std::max_element(inb.begin(), inb.end()) + 0.5 * *std::max_element(outb.begin(), outb.end()) + 3.0 * imb;
    };
    unsigned long long rng = 0x9E3779B97F4A7C15ull;
    auto next = [&]() { rng = rng * 6364136223846793005ull + 1442695040888963407ull; return (unsigned)(rng >> 33); };
    double cur = cost(), best = cur, T = 3.0;
    std::vector<uint8_t> best_owner = owner;
    const int iters = 40000;
    for (int it = 0; it < iters; it++) {
        const int a = (int)(next() % (unsigned)ncell);
        double c;
        int b = -1;
        uint8_t olda = owner[a];
        if (next() & 1u) {
            const uint8_t nw = (uint8_t)(next() % (unsigned)world);
            if (nw == olda) continue;
            owner[a] = nw;
        } else {
            b = (int)(next() % (unsigned)ncell);
            if (owner[b] == olda) continue;
            std::swap(owner[a], owner[b]);
        }
        c = cost();
        // accept improvements always, deteriorations with probability 2^(-(c - cur) / T) (integer-only randomness: deterministic)
        bool accept = c <= cur;
        if (!accept) {
            const double x = (c - cur) / T;
            accept = x < 30.0 && (double)(next() & 0xFFFFFF) / 16777216.0 < exp2(-x);
        }
        if (accept) {
            cur = c;
            if (cur < best) { best = cur; best_owner = owner; }
        } else if (b >= 0) {
            std::swap(owner[a], owner[b]);
        } else {
            owner[a] = olda;
        }
        T = std::max(0.05, T * 0.9997);
    }
    owner = best_owner;
    if (getenv("KP_SHARD_VERBOSE")) {
        cost();
        fprintf(stderr, "kp_shard: %d x %d cells over %d ranks: busiest rank receives %d cells, sends %d; cost %.2f -> %.2f\n", r1, r2, world,
                *std::max_element(inb.begin(), inb.end()), *std::max_element(outb.begin(), outb.end()), cost(), best);
    }
}

// digits of the top position dealt round-robin in order of decreasing level: every rank gets a similar mix of
// levels (= a similar share of every wave) and a similar number of splits
static int shard_assignment(const kp_plan *p, int world, uint8_t *owner, uint8_t *slot, uint32_t *nslots_of_rank)
{
    const KpTables &t = p->host.t;
    if (t.nhigh < 1) return fail("sharding needs at least one high position (the pattern is too small to shard)");
    const int e = t.highpos[t.nhigh - 1];
    const int radix = t.radix[e];
    if (world < 1 || world > KP_MAX_SHARDS || world > radix) return fail("sharding: world size must be 1..min(8, radix of the top position)");
    std::vector<int> digits(radix);
    for (int d = 0; d < radix; d++) digits[d] = d;
    auto lvl = [&](int d) { unsigned m = t.digit_mask[e][d]; return (int)((m & 1) + ((m >> 1) & 1) + ((m >> 2) & 1) + ((m >> 3) & 1)); };
    std::stable_sort(digits.begin(), digits.end(), [&](int a, int b) { return lvl(a) > lvl(b); });
    for (int r = 0; r < KP_MAX_SHARDS; r++) nslots_of_rank[r] = 0;
    memset(owner, 0, 16);
    memset(slot, 0, 16);
    for (int i = 0; i < radix; i++) {
        const int r = i % world, d = digits[i];
        owner[d] = (uint8_t)r;
        slot[d] = (uint8_t)nslots_of_rank[r]++;
    }
    return 0;
}

int kp_shard_assignment(const kp_plan *p, int world, uint8_t *owner16, uint8_t *slot16)
{
    if (!p || !owner16 || !slot16) return fail("kp_shard_assignment: null argument");
    uint32_t n[KP_MAX_SHARDS];
    return shard_assignment(p, world, owner16, slot16, n);
}

int kp_shard_create(kp_plan *p, int rank, int world, int replicate, kp_shard **out)
{
    if (!p || !out) return fail("kp_shard_create: null argument");
    if (!p->host.lattice) return fail("kp_shard_create: this plan was created without the tile lattice (kp_plan_create_lite)");
    const KpTables &t = p->host.t;
    if (t.r0 != 15) return fail("kp_shard_create: the sharded DP needs an N position in the general pattern");
    if (rank < 0 || rank >= world) return fail("kp_shard_create: bad rank");
    KP_CUDA(cudaSetDevice(p->device));
    kp_shard *s = new kp_shard();
    uint32_t nslots[KP_MAX_SHARDS];
    memset(&s->view, 0, sizeof s->view);
    if (shard_assignment(p, world, s->view.owner, s->view.slot, nslots)) { delete s; return 1; }
    const int e = t.highpos[t.nhigh - 1];
    s->plan = p; s->rank = rank; s->world = world; s->replicate = replicate != 0;
    s->hw_top = t.highw[e]; s->radix_top = t.radix[e]; s->nslots = nslots[rank];
    s->view.hw_top = s->hw_top;
    const uint64_t own_tiles = (uint64_t)s->nslots * s->hw_top;
    s->local_tiles = own_tiles;
    std::vector<uint8_t> cell_owner;   // two-dimensional ownership: owner of every (top digit, second digit) cell
    if (s->replicate) {   // full-size table, global tile numbers; readers of a digit = owners of its strict supersets
        s->local_tiles = t.ntiles;
        for (int d = 0; d < (int)s->radix_top; d++) {
            s->view.slot[d] = (uint8_t)d;
            unsigned mask = 0;
            for (int q = 0; q < (int)s->radix_top; q++) {
                const unsigned md = t.digit_mask[e][d], mq = t.digit_mask[e][q];
                if (q != d && (md & mq) == md && s->view.owner[q] != s->view.owner[d]) mask |= 1u << s->view.owner[q];
            }
            s->view.push_mask[d] = (uint8_t)mask;
        }
        if (t.nhigh >= 2 && world > 1 && !getenv("KP_SHARD_1D")) {
            // Two-dimensional ownership over the two top high positions: cell (d_top, d_second) belongs to rank
            // (i_top + i_second) mod world, i = index of the digit in order of decreasing level.  Every wave (= level)
            // is spread over all ranks, and so is the traffic: a tile is pushed to the owners of its parents along BOTH
            // positions (about four peers at eight ranks), but no rank receives more than its share.
            const int e2 = t.highpos[t.nhigh - 2];
            const int r1 = t.radix[e], r2 = t.radix[e2];
            auto level_index = [&](int pos, std::vector<int> &idx) {
                const int radix = t.radix[pos];
                std::vector<int> digits(radix);
                for (int d = 0; d < radix; d++) digits[d] = d;
                auto lvl = [&](int d) { unsigned m = t.digit_mask[pos][d]; return (int)((m & 1) + ((m >> 1) & 1) + ((m >> 2) & 1) + ((m >> 3) & 1)); };
                std::stable_sort(digits.begin(), digits.end(), [&](int a, int b) { return lvl(a) > lvl(b); });
                idx.assign(radix, 0);
                for (int i = 0; i < radix; i++) idx[digits[i]] = i;
            };
            std::vector<int> i1, i2;
            level_index(e, i1);
            level_index(e2, i2);
            s->view.two_d = 1;
            s->view.hw_second = t.highw[e2];
            cell_owner.assign((size_t)r1 * r2, 0);
            for (int d1 = 0; d1 < r1; d1++)
                for (int d2 = 0; d2 < r2; d2++) cell_owner[(size_t)d2 + (size_t)r2 * d1] = (uint8_t)((i1[d1] + i2[d2]) % world);
            if (world > 1 && !getenv("KP_SHARD_MODULAR")) {
                if (r1 == 15 && r2 == 15 && world <= 8 && !getenv("KP_SHARD_SEARCH")) {
                    // two N positions: tables found offline by a longer run of the same search (tools/optimise_shard_owners.py)
                    for (int d1 = 0; d1 < 15; d1++)
                        for (int d2 = 0; d2 < 15; d2++) cell_owner[(size_t)d2 + 15u * d1] = kp_shard_owner_tab[world - 2][d1][d2];
                } else {
                    optimise_cell_owners(t, e, e2, world, cell_owner);
                }
            }
            for (int d1 = 0; d1 < r1; d1++)
                for (int d2 = 0; d2 < r2; d2++) {
                    const size_t c = (size_t)d2 + (size_t)r2 * d1;
                    unsigned mask = 0;
                    for (int q = 0; q < r1; q++) {
                        const unsigned md = t.digit_mask[e][d1], mq = t.digit_mask[e][q];
                        if (q != d1 && (md & mq) == md) mask |= 1u << cell_owner[(size_t)d2 + (size_t)r2 * q];
                    }
                    for (int q = 0; q < r2; q++) {
                        const unsigned md = t.digit_mask[e2][d2], mq = t.digit_mask[e2][q];
                        if (q != d2 && (md & mq) == md) mask |= 1u << cell_owner[(size_t)q + (size_t)r2 * d1];
                    }
                    mask &= ~(1u << cell_owner[c]);
                    s->view.owner2[c] = cell_owner[c];
                    s->view.push_mask2[c] = (uint8_t)mask;
                }
            uint32_t cells = 0;
            for (uint8_t o : cell_owner) cells += o == rank;
            s->nslots = cells;   // reported as top_digits: the number of (top, second) cells this rank owns
        }
    }
    if (s->local_tiles >= (1ull << 28)) { delete s; return fail("kp_shard_create: more than 2^28 tiles per rank"); }
    // this rank's tiles of every wave, in the order of the plan's tile list
    const size_t nhl = p->host.hl_off.size() - 1;
    std::vector<uint32_t> mine;
    s->hl_off.assign(nhl + 1, 0);
    for (size_t l = 0; l < nhl; l++) {
        for (uint64_t i = p->host.hl_off[l]; i < p->host.hl_off[l + 1]; i++) {
            const uint32_t tile = p->host.tile_order[i];
            const int own = s->view.two_d ? cell_owner[tile / s->view.hw_second] : s->view.owner[tile / s->hw_top];
            if (own == rank) mine.push_back(tile);
        }
        s->hl_off[l + 1] = mine.size();
    }
    if (!s->view.two_d && mine.size() != own_tiles) { delete s; return fail("kp_shard_create: internal: tile count"); }
    cudaError_t e1 = cudaMalloc(&s->d_best, (size_t)s->local_tiles * t.tile_stride * sizeof(float));
    cudaError_t e2 = cudaMalloc(&s->d_kept, (size_t)s->local_tiles * t.rp * sizeof(uint16_t));
    cudaError_t e3 = cudaMalloc(&s->d_tiles, sizeof(uint32_t) * (mine.size() + 1));
    cudaError_t e4 = cudaMalloc(&s->d_counters, sizeof(uint32_t) * 64);
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess || e4 != cudaSuccess) {
        cudaFree(s->d_best); cudaFree(s->d_kept); cudaFree(s->d_tiles); cudaFree(s->d_counters);
        delete s;
        cudaGetLastError();
        return fail("kp_shard_create: out of device memory for the shard");
    }
    KP_CUDA(cudaMemcpy(s->d_tiles, mine.data(), sizeof(uint32_t) * mine.size(), cudaMemcpyHostToDevice));
    s->view.best[rank] = s->d_best;
    s->view.flags[rank] = s->d_kept;
    KP_CUDA(cudaFuncSetAttribute(dp_kernel_sharded<true, 1>(t.rp), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem_optin));
    KP_CUDA(cudaFuncSetAttribute(dp_kernel_sharded<false, 1>(t.rp), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem_optin));
    KP_CUDA(cudaFuncSetAttribute(dp_kernel_sharded<true, 2>(t.rp), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem_optin));
    KP_CUDA(cudaFuncSetAttribute(dp_kernel_sharded<false, 2>(t.rp), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem_optin));
    *out = s;
    return 0;
}

int kp_shard_destroy(kp_shard *s)
{
    if (!s) return 0;
    cudaSetDevice(s->plan->device);
    cudaFree(s->d_best); cudaFree(s->d_kept); cudaFree(s->d_tiles); cudaFree(s->d_counters);
    delete s;
    return 0;
}

int kp_shard_get_info(const kp_shard *s, kp_shard_info *o)
{
    if (!s || !o) return fail("kp_shard_get_info: null argument");
    const KpTables &t = s->plan->host.t;
    o->local_tiles = s->local_tiles;
    o->table_elems = s->local_tiles * t.tile_stride;
    o->kept_elems = s->local_tiles * (uint64_t)t.rp;
    o->d_best = (uint64_t)(uintptr_t)s->d_best;
    o->d_kept = (uint64_t)(uintptr_t)s->d_kept;
    o->rank = (uint32_t)s->rank;
    o->world = (uint32_t)s->world;
    o->nwaves = (uint32_t)(s->hl_off.size() - 1);
    o->top_digits = s->nslots;
    o->replicate = s->replicate ? 1u : 0u;
    return 0;
}

int kp_shard_set_peer(kp_shard *s, int peer, const float *d_best, const uint16_t *d_kept)
{
    if (!s || peer < 0 || peer >= s->world || !d_best || !d_kept) return fail("kp_shard_set_peer: bad argument");
    if (peer == s->rank) return fail("kp_shard_set_peer: peer is this rank");
    s->view.best[peer] = d_best;
    s->view.flags[peer] = d_kept;
    return 0;
}

// CUDA IPC plumbing for one-process-per-GPU launches: export a device allocation, map a peer's
int kp_ipc_export(const void *d_ptr, uint8_t *handle64)
{
    if (!d_ptr || !handle64) return fail("kp_ipc_export: null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    KP_CUDA(cudaIpcGetMemHandle(&h, (void *)d_ptr));
    memcpy(handle64, &h, 64);
    return 0;
}

int kp_ipc_open(int device, const uint8_t *handle64, void **d_ptr)
{
    if (!handle64 || !d_ptr) return fail("kp_ipc_open: null argument");
    KP_CUDA(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    KP_CUDA(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}

int kp_ipc_close(int device, void *d_ptr)
{
    if (!d_ptr) return 0;
    KP_CUDA(cudaSetDevice(device));
    KP_CUDA(cudaIpcCloseMemHandle(d_ptr));
    return 0;
}

// one wave of this rank's tiles on the counts d_expM - d_subM, d_expU - d_subU (d_sub*: null for none, as in dp_counts)
static int shard_wave(kp_shard *s, int wave, const int64_t *d_expM, const int64_t *d_expU, const int64_t *d_subM,
                      const int64_t *d_subU, uint64_t max_count, double alpha, double beta, double penalty, void *stream,
                      const char *what)
{
    if (!s) return fail(std::string(what) + ": null shard");
    kp_plan *p = s->plan;
    const KpTables &t = p->host.t;
    if (wave < 0 || wave >= (int)s->hl_off.size() - 1 || wave >= 64) return fail(std::string(what) + ": bad wave");
    for (int r = 0; r < s->world; r++)
        if (!s->view.best[r] || !s->view.flags[r]) return fail(std::string(what) + ": a peer's shard has not been set");
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    if (wave == 0) KP_CUDA(cudaMemsetAsync(s->d_counters, 0, sizeof(uint32_t) * 64, st));
    const uint64_t lo = s->hl_off[wave], hi = s->hl_off[wave + 1];
    if (hi == lo) return 0;
    const bool wide = max_count > 0xFFFFFFFFull;
    const int nw = p->nwarps[wide];
    if (nw < 1) return fail("DP kernel does not fit in shared memory for this tile shape");
    KpDpParams prm;
    memset(&prm, 0, sizeof prm);
    prm.tab = p->d_tab;
    prm.rowtab = p->d_rowtab;
    prm.e0 = (const long long *)d_expM;
    prm.e1 = (const long long *)d_expU;
    prm.s0 = (const long long *)d_subM;
    prm.s1 = (const long long *)d_subU;
    prm.alpha = alpha; prm.beta = beta; prm.penalty = penalty;
    prm.best = s->d_best;
    prm.flags = s->d_kept;
    prm.pf_dist = p->pf_dist;
    prm.view = s->view;
    prm.my_rank = s->rank;
    prm.tile_list = s->d_tiles + lo;
    prm.ntiles_wave = (uint32_t)(hi - lo);
    prm.counter = s->d_counters + wave;
    prm.leaf_wave = (wave == 0);
    const uint64_t ntile = hi - lo;
    int warps = nw;
    if (ntile < (uint64_t)p->sm_count * nw) {
        warps = (int)((ntile + p->sm_count - 1) / p->sm_count);
        if (warps < 1) warps = 1;
    }
    uint64_t grid = (ntile + warps - 1) / warps;
    if (grid > (uint64_t)p->sm_count) grid = p->sm_count;
    const size_t sm = 2048 + t.rt_bytes + (size_t)warps * t.warp_smem_bytes[wide];
    if (s->replicate) {
        if (t.rp == KP_RP_NN) launch_dp_r0<15, KP_RP_NN, 2>(wide, (int)grid, warps * 32, sm, st, prm);
        else launch_dp_r0<15, 0, 2>(wide, (int)grid, warps * 32, sm, st, prm);
    } else {
        if (t.rp == KP_RP_NN) launch_dp_r0<15, KP_RP_NN, 1>(wide, (int)grid, warps * 32, sm, st, prm);
        else launch_dp_r0<15, 0, 1>(wide, (int)grid, warps * 32, sm, st, prm);
    }
    p->launches++;
    KP_CUDA(cudaGetLastError());
    return 0;
}

int kp_shard_dp_wave(kp_shard *s, int wave, const int64_t *d_expM, const int64_t *d_expU, uint64_t max_count, double alpha,
                     double beta, double penalty, void *stream)
{
    return shard_wave(s, wave, d_expM, d_expU, nullptr, nullptr, max_count, alpha, beta, penalty, stream, "kp_shard_dp_wave");
}

int kp_shard_cv_wave(kp_shard *s, int wave, const int64_t *d_expMtot, const int64_t *d_expUtot, const int64_t *d_expMtest,
                     const int64_t *d_expUtest, uint64_t max_count, double alpha, double beta_fold, double penalty, void *stream)
{
    if (!d_expMtest || !d_expUtest) return fail("kp_shard_cv_wave: null held-out table");
    return shard_wave(s, wave, d_expMtot, d_expUtot, d_expMtest, d_expUtest, max_count, alpha, beta_fold, penalty, stream,
                      "kp_shard_cv_wave");
}

// kp_cv_heldout over the shard view: the backtrack reads the peers' tables, the leaf kernel this rank's (replicated) count
// tables; the root's train loss comes from the same device gather as kp_shard_gather
int kp_shard_cv_heldout(kp_shard *s, const int64_t *d_expMtot, const int64_t *d_expUtot, const int64_t *d_expMtest,
                        const int64_t *d_expUtest, double alpha, double beta_fold, double penalty, uint64_t root, void *d_ws,
                        uint64_t cap, float *h_top, void *stream)
{
    if (!s || !d_expMtot || !d_expUtot || !d_expMtest || !d_expUtest || !d_ws || !h_top)
        return fail("kp_shard_cv_heldout: null argument");
    kp_plan *p = s->plan;
    if (p->host.t.total_level > 64) return fail("kp_shard_cv_heldout: more than 64 levels");
    if (root == UINT64_MAX) root = p->host.npat - 1;
    if (root >= p->host.npat) return fail("kp_shard_cv_heldout: root out of range");
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    if (scratch_reserve(p, sizeof(float), st)) return 1;
    float *d_rootval = (float *)p->d_scratch;
    unsigned long long *sorted, *keys, *ctr;
    float *vals;
    if (backtrack_device(p, s->view, d_ws, cap, root, st, &sorted, &keys, &vals, &ctr)) return 1;
    kp_cv_leaf_kernel<<<p->sm_count, 128, 0, st>>>(p->d_tab, p->d_rowtab, (const long long *)d_expMtot, (const long long *)d_expUtot,
                                                   (const long long *)d_expMtest, (const long long *)d_expUtest, alpha, beta_fold,
                                                   penalty, sorted, ctr, cap, vals);
    kp_gather_kernel<<<1, 32, 0, st>>>(p->d_tab, p->d_rowtab, s->view, nullptr, root, 1, d_rootval);
    p->launches += 2;
    KP_CUDA(cudaGetLastError());
    unsigned long long hc[2] = {0, 0};
    int herr = 0;
    float htrain = 0.f;
    KP_CUDA(cudaMemcpyAsync(hc, ctr, sizeof hc, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaMemcpyAsync(&herr, p->d_err, sizeof herr, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaMemcpyAsync(&htrain, d_rootval, sizeof htrain, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    if (herr == 2) return fail("kp_shard_cv_heldout: the DP gave up waiting for a child tile (internal error)");
    if (hc[1] || hc[0] > cap) return fail_capacity("kp_shard_cv_heldout: partition larger than the workspace capacity");
    if (hc[0] == 0) return fail("kp_shard_cv_heldout: the backtrack produced no leaf (internal error)");
    std::vector<unsigned long long> hk(hc[0]);
    std::vector<float> hv(hc[0]);
    KP_CUDA(cudaMemcpyAsync(hk.data(), keys, hc[0] * 8, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaMemcpyAsync(hv.data(), vals, hc[0] * 4, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    h_top[0] = htrain;
    h_top[1] = tree_sum(hk.data(), hv.data(), 0, hc[0], 0);
    return 0;
}

int kp_shard_backtrack(kp_shard *s, void *d_ws, uint64_t cap, uint64_t root, uint64_t *h_patnums, uint64_t *n_out, void *stream)
{
    if (!s || !d_ws || !h_patnums || !n_out) return fail("kp_shard_backtrack: null argument");
    kp_plan *p = s->plan;
    if (root == UINT64_MAX) root = p->host.npat - 1;
    if (root >= p->host.npat) return fail("kp_shard_backtrack: root out of range");
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    unsigned long long *sorted, *keys, *ctr;
    float *vals;
    if (backtrack_device(p, s->view, d_ws, cap, root, st, &sorted, &keys, &vals, &ctr)) return 1;
    unsigned long long hc[2] = {0, 0};
    KP_CUDA(cudaMemcpyAsync(hc, ctr, sizeof hc, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    *n_out = hc[0];
    if (hc[1] || hc[0] > cap) return fail_capacity("kp_shard_backtrack: partition larger than the workspace capacity");
    KP_CUDA(cudaMemcpyAsync(h_patnums, sorted, hc[0] * 8, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// scores / kept-whole flags / split codes of arbitrary patterns, read through the view (any rank's shard)
int kp_shard_gather(kp_shard *s, const uint64_t *h_patnums, uint64_t n, float *h_best, uint8_t *h_kept, uint8_t *h_codes,
                    void *stream)
{
    if (!s || !h_patnums) return fail("kp_shard_gather: null argument");
    if (n == 0) return 0;
    kp_plan *p = s->plan;
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    if (scratch_reserve(p, n * 16, st)) return 1;
    unsigned long long *d_pat = (unsigned long long *)p->d_scratch;
    float *d_val = (float *)(d_pat + n);
    uint8_t *d_k = (uint8_t *)(d_val + n), *d_c = d_k + n;
    KP_CUDA(cudaMemcpyAsync(d_pat, h_patnums, n * 8, cudaMemcpyHostToDevice, st));
    const int grid = grid_for(n, 256, p->sm_count);
    if (h_best) kp_gather_kernel<<<grid, 256, 0, st>>>(p->d_tab, p->d_rowtab, s->view, d_pat, 0, n, d_val);
    if (h_kept) kp_gather_flags_kernel<<<grid, 256, 0, st>>>(p->d_tab, p->d_rowtab, s->view, d_pat, 0, n, d_k);
    if (h_codes) kp_split_codes_kernel<<<grid, 256, 0, st>>>(p->d_tab, p->d_rowtab, s->view, d_pat, n, d_c);
    KP_CUDA(cudaGetLastError());
    if (h_best) KP_CUDA(cudaMemcpyAsync(h_best, d_val, n * 4, cudaMemcpyDeviceToHost, st));
    if (h_kept) KP_CUDA(cudaMemcpyAsync(h_kept, d_k, n, cudaMemcpyDeviceToHost, st));
    if (h_codes) KP_CUDA(cudaMemcpyAsync(h_codes, d_c, n, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// float64 sum of the leaves' losses in the order of the recursion (s1 + s2 at every inner node; keys sorted ascending)
static double tree_sum_f64(const KpGreedyLeaf *lv, size_t lo, size_t hi, int depth)
{
    if (hi - lo == 1) return lv[lo].loss;
    const unsigned long long bit = 1ULL << (63 - depth);
    size_t a = lo, b = hi;
    while (a < b) {
        size_t mid = (a + b) / 2;
        if (lv[mid].key & bit) b = mid; else a = mid + 1;
    }
    if (a == lo || a == hi) return tree_sum_f64(lv, lo, hi, depth + 1);
    volatile double l = tree_sum_f64(lv, lo, a, depth + 1), r = tree_sum_f64(lv, a, hi, depth + 1);
    volatile double sum = l + r;
    return sum;
}

uint64_t kp_greedy_ws_bytes(uint64_t cap)
{
    return 2 * cap * sizeof(KpBtNode) + 2 * cap * sizeof(KpGreedyLeaf) + 80 * 8 + cap * KP_GREEDY_ACC * 8 + 2 * cap * 8 + 64;
}

int kp_greedy(kp_plan *p, const int64_t *d_kmerM, const int64_t *d_kmerU, const int64_t *d_testM, const int64_t *d_testU,
              double alpha, double beta, double penalty, void *d_ws, uint64_t cap, uint64_t *h_patnums, double *h_loss,
              double *h_test, uint64_t *n_out, double *h_total, void *stream)
{
    if (!p || !d_kmerM || !d_kmerU || !d_ws || !h_patnums || !n_out) return fail("kp_greedy: null argument");
    if ((d_testM == nullptr) != (d_testU == nullptr)) return fail("kp_greedy: give both held-out tables or none");
    if (p->host.t.total_level > 63) return fail("kp_greedy: more than 63 levels");
    cudaStream_t st = (cudaStream_t)stream;
    KP_CUDA(cudaSetDevice(p->device));
    KpBtNode *fa = (KpBtNode *)d_ws, *fb = fa + cap;
    KpGreedyLeaf *leaves = (KpGreedyLeaf *)(fb + cap), *sorted = leaves + cap;
    unsigned long long *ctr = (unsigned long long *)(sorted + cap);
    unsigned long long *acc = ctr + 80;
    unsigned long long *sa = acc + cap * KP_GREEDY_ACC, *sb = sa + cap;   // k-mers per frontier node
    kp_backtrack_init_kernel<<<1, 128, 0, st>>>(fa, p->host.npat - 1, ctr);
    kp_greedy_init_kernel<<<1, 1, 0, st>>>(sa, p->host.nkmer);
    KP_CUDA(cudaMemsetAsync(acc, 0, cap * KP_GREEDY_ACC * 8, st));
    const int levels = (int)p->host.t.total_level + 1;
    const int grid = p->sm_count * 4;
    const unsigned long long big = 32768;   // nodes with at least this many k-mers are shared by all CTAs
    for (int d = 0; d < levels && d < 64; d++) {
        kp_greedy_marginals_kernel<<<grid, 256, 0, st>>>(p->d_tab, (const long long *)d_kmerM, (const long long *)d_kmerU,
                                                         (const long long *)d_testM, (const long long *)d_testU, d,
                                                         (d & 1) ? fb : fa, (d & 1) ? sb : sa, ctr, big, cap, acc);
        kp_greedy_decide_kernel<<<grid, 256, 0, st>>>(p->d_tab, d_testM != nullptr, alpha, beta, penalty, d, (d & 1) ? fb : fa,
                                                      (d & 1) ? sb : sa, (d & 1) ? fa : fb, (d & 1) ? sa : sb, leaves, cap, ctr,
                                                      acc);
        p->launches += 2;
    }
    kp_greedy_sort_kernel<<<p->sm_count, 256, 0, st>>>(leaves, ctr, cap, sorted);
    p->launches += 2;
    KP_CUDA(cudaGetLastError());
    unsigned long long hc[2] = {0, 0};
    KP_CUDA(cudaMemcpyAsync(hc, ctr, sizeof hc, cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    *n_out = hc[0];
    if (hc[1] || hc[0] > cap) return fail_capacity("kp_greedy: partition larger than the workspace capacity");
    if (hc[0] == 0) return fail("kp_greedy: no leaf (internal error)");
    std::vector<KpGreedyLeaf> hv(hc[0]);
    KP_CUDA(cudaMemcpyAsync(hv.data(), sorted, hc[0] * sizeof(KpGreedyLeaf), cudaMemcpyDeviceToHost, st));
    KP_CUDA(cudaStreamSynchronize(st));
    for (size_t i = 0; i < hv.size(); i++) {
        h_patnums[i] = hv[i].pat;
        if (h_loss) h_loss[i] = hv[i].loss;
        if (h_test) h_test[i] = hv[i].test;
    }
    if (h_total) *h_total = tree_sum_f64(hv.data(), 0, hv.size(), 0);
    return 0;
}

int kp_kmer_fold_terms(int device, const int64_t *h_Mtr, const int64_t *h_Utr, const int64_t *h_Mte, const int64_t *h_Ute,
                       const double *h_beta, uint64_t n, double alpha, double *h_train, double *h_test)
{
    if (!h_Mtr || !h_Utr || !h_Mte || !h_Ute || !h_beta || !h_train || !h_test) return fail("kp_kmer_fold_terms: null argument");
    if (n == 0) return 0;
    KP_CUDA(cudaSetDevice(device));
    long long *d_in = nullptr;
    double *d_f = nullptr;
    KP_CUDA(cudaMalloc(&d_in, n * 8 * 4));
    cudaError_t e = cudaMalloc(&d_f, n * 8 * 3);
    if (e != cudaSuccess) { cudaFree(d_in); return fail("kp_kmer_fold_terms: out of device memory"); }
    const int64_t *src[4] = {h_Mtr, h_Utr, h_Mte, h_Ute};
    for (int i = 0; i < 4; i++) cudaMemcpy(d_in + i * n, src[i], n * 8, cudaMemcpyHostToDevice);
    cudaMemcpy(d_f, h_beta, n * 8, cudaMemcpyHostToDevice);
    kp_kmer_fold_terms_kernel<<<296, 256>>>(d_in, d_in + n, d_in + 2 * n, d_in + 3 * n, d_f, n, alpha, d_f + n, d_f + 2 * n);
    cudaError_t e2 = cudaGetLastError();
    cudaMemcpy(h_train, d_f + n, n * 8, cudaMemcpyDeviceToHost);
    cudaError_t e3 = cudaMemcpy(h_test, d_f + 2 * n, n * 8, cudaMemcpyDeviceToHost);
    cudaFree(d_in);
    cudaFree(d_f);
    if (e2 != cudaSuccess || e3 != cudaSuccess) return fail(std::string("kp_kmer_fold_terms: ") + cudaGetErrorString(e2 != cudaSuccess ? e2 : e3));
    return 0;
}

int kp_debug_log(int device, const double *h_x, double *h_y, uint64_t n)
{
    KP_CUDA(cudaSetDevice(device));
    double *dx = nullptr, *dy = nullptr;
    KP_CUDA(cudaMalloc(&dx, n * 8));
    KP_CUDA(cudaMalloc(&dy, n * 8));
    KP_CUDA(cudaMemcpy(dx, h_x, n * 8, cudaMemcpyHostToDevice));
    kp_debug_log_kernel<<<296, 256>>>(dx, dy, n);
    KP_CUDA(cudaGetLastError());
    KP_CUDA(cudaMemcpy(h_y, dy, n * 8, cudaMemcpyDeviceToHost));
    cudaFree(dx);
    cudaFree(dy);
    return 0;
}

int kp_debug_leaf_score(int device, const int64_t *h_M, const int64_t *h_U, uint64_t n, double alpha, double beta,
                        double penalty, double *h_out)
{
    KP_CUDA(cudaSetDevice(device));
    long long *dm = nullptr, *du = nullptr;
    double *dout = nullptr;
    KP_CUDA(cudaMalloc(&dm, n * 8));
    KP_CUDA(cudaMalloc(&du, n * 8));
    KP_CUDA(cudaMalloc(&dout, n * 8));
    KP_CUDA(cudaMemcpy(dm, h_M, n * 8, cudaMemcpyHostToDevice));
    KP_CUDA(cudaMemcpy(du, h_U, n * 8, cudaMemcpyHostToDevice));
    kp_debug_leaf_kernel<<<296, 256>>>(dm, du, n, alpha, beta, penalty, dout);
    KP_CUDA(cudaGetLastError());
    KP_CUDA(cudaMemcpy(h_out, dout, n * 8, cudaMemcpyDeviceToHost));
    cudaFree(dm);
    cudaFree(du);
    cudaFree(dout);
    return 0;
}

int kp_debug_self_score(int device, const int64_t *h_M, const int64_t *h_U, const double *h_alpha, const double *h_beta,
                        const double *h_penalty, const uint8_t *h_wide, uint64_t n, float *h_lb, uint8_t *h_ok, float *h_sf,
                        uint8_t *h_rup, double *h_fast, double *h_exact)
{
    if (!h_M || !h_U || !h_alpha || !h_beta || !h_penalty || !h_wide || !h_lb || !h_ok || !h_sf || !h_rup || !h_fast || !h_exact)
        return fail("kp_debug_self_score: null argument");
    if (n == 0) return 0;
    for (uint64_t i = 0; i < n; i++) {
        uint64_t tot = 0;
        for (int b = 0; b < 8; b++) {
            const int64_t c = b < 4 ? h_M[4 * i + b] : h_U[4 * i + b - 4];
            if (c < 0) return fail("kp_debug_self_score: negative count");
            tot += (uint64_t)c;
            if (tot >> 62) return fail("kp_debug_self_score: counts of an item sum to 2^62 or more");
        }
        if (!h_wide[i] && (tot >> 32)) return fail("kp_debug_self_score: narrow (32-bit) item whose counts sum to 2^32 or more");
    }
    KP_CUDA(cudaSetDevice(device));
    // inputs: M, U (8 x 8 bytes), alpha, beta, penalty (3 x 8), wide (1); outputs: st, exact (2 x 8), lb, sf (2 x 4), ok, rup (2)
    const size_t per = 8 * 8 + 3 * 8 + 1 + 2 * 8 + 2 * 4 + 2;
    unsigned char *d = nullptr;
    KP_CUDA(cudaMalloc(&d, n * per));
    long long *dM = (long long *)d, *dU = dM + 4 * n;
    double *da = (double *)(dU + 4 * n), *db = da + n, *dp = db + n, *dst = dp + n, *dex = dst + n;
    float *dlb = (float *)(dex + n), *dsf = dlb + n;
    unsigned char *dw = (unsigned char *)(dsf + n), *dok = dw + n, *drup = dok + n;
    cudaMemcpy(dM, h_M, n * 32, cudaMemcpyHostToDevice);
    cudaMemcpy(dU, h_U, n * 32, cudaMemcpyHostToDevice);
    cudaMemcpy(da, h_alpha, n * 8, cudaMemcpyHostToDevice);
    cudaMemcpy(db, h_beta, n * 8, cudaMemcpyHostToDevice);
    cudaMemcpy(dp, h_penalty, n * 8, cudaMemcpyHostToDevice);
    cudaError_t e = cudaMemcpy(dw, h_wide, n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        kp_debug_self_score_kernel<<<296, 256>>>(dM, dU, da, db, dp, dw, n, dlb, dok, dsf, drup, dst, dex);
        e = cudaGetLastError();
    }
    const void *src[6] = {dlb, dok, dsf, drup, dst, dex};
    void *dst_h[6] = {h_lb, h_ok, h_sf, h_rup, h_fast, h_exact};
    const size_t bytes[6] = {4, 1, 4, 1, 8, 8};
    for (int k = 0; k < 6 && e == cudaSuccess; k++) e = cudaMemcpy(dst_h[k], src[k], n * bytes[k], cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) return fail(std::string("kp_debug_self_score: ") + cudaGetErrorString(e));
    return 0;
}

}  // extern "C"
