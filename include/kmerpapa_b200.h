/*
 * kmerpapa_b200.h — C ABI of libkpapa.so, the B200 (sm_100a) implementation of kmerPaPa's
 * optimal k-mer pattern-partition dynamic program.
 *
 * The reference (BesenbacherLab/kmerPaPa v0.2.4) is pure Python + numba and has no FFI layer; its
 * drop-in boundary is the pair of Python functions cli.py calls.  Each entry point below names
 * the reference code it replaces (paths relative to the reference checkout):
 *
 *   kp_pack_counts     src/kmerpapa/io_utils.py:82-136 (read_dict dedup/sum) +
 *                      src/kmerpapa/algorithms/bottum_up_array_w_numba.py:106-114 (level-0 fill)
 *   kp_expand_counts   bottum_up_array_w_numba.py:50-53 and
 *                      bottum_up_array_penalty_plus_pseudo_CV.py:52-59 (pattern counts = sum of two
 *                      disjoint sub-patterns; train = total - held-out)
 *   kp_dp_single       bottum_up_array_w_numba.py:26-64,116-120 (score + min-plus recurrence)
 *   kp_backtrack       bottum_up_array_w_numba.py:8-24 (DFS, c1 subtree first)
 *   kp_split_codes     the backtrack_mem entry of bottum_up_array_w_numba.py:48-49, :64
 *   kp_dp_cv_job       bottum_up_array_penalty_plus_pseudo_CV.py:15-78,145-157, one fold per call
 *   kp_cv_heldout      the test_score_mem entry of ..._CV.py:46-51, :71-78
 *   kp_pattern_counts  src/kmerpapa/pattern_utils.py:192-215 (get_M_U, used by cli.py:281-283)
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error; kp_last_error() gives the message
 *     (thread-local).  No function falls back to a CPU path: without a usable CUDA device the
 *     plan cannot be created and everything else fails.
 *   - d_* are device pointers owned by the caller (the Python host allocates them as torch
 *     tensors), h_* are host pointers.  `stream` is a cudaStream_t passed as void*.
 *   - score tables live in a tiled device layout (kmerpapa_b200/csrc/kp_tables.h): the pattern table is
 *     cut into tiles over a subset of positions, rows of a tile are stored in schedule order.  The
 *     reference's dense pattern number (pattern_utils.py:237-257) is the external numbering everywhere
 *     in this API; kp_gather_table / kp_gather_kept / kp_split_codes translate.
 *   - a plan is bound to one device and one general pattern; it is not thread-safe, different
 *     plans may be used from different threads.
 */
#ifndef KMERPAPA_B200_H
#define KMERPAPA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct kp_plan kp_plan;

typedef struct kp_plan_info {
    uint64_t npat;           /* number of patterns = prod radix_i (pattern_utils.py:587-599) */
    uint64_t nkmer;          /* number of k-mers matched by the general pattern */
    uint64_t ntiles;         /* npat / tile_cells */
    uint64_t table_elems;    /* ntiles * tile_stride: float elements of d_best / d_train / d_test */
    uint64_t kept_elems;     /* ntiles * rows (padded): uint16 elements of d_kept */
    uint64_t expanded_elems; /* ntiles * tile_kmers: elements of each expanded count table */
    uint64_t backtrack_ws_bytes; /* bytes of device workspace kp_backtrack needs for `cap` = 65536 */
    uint32_t k;              /* pattern length */
    uint32_t nlevels;        /* pattern_level(gen_pat) + 1 */
    uint32_t tile_cells;     /* patterns per tile (product of the radices of the on-chip positions) */
    uint32_t tile_stride;    /* tile pitch in float elements */
    uint32_t tile_kmers;     /* k-mers spanned by the on-chip positions */
    uint32_t low_positions;  /* number of (non-fixed) positions kept on chip */
    uint32_t register_radix; /* radix of the position held in registers (15 for N) */
    uint32_t rows, rounds;   /* rows per tile and rounds of the row schedule */
    uint32_t warps_per_cta;  /* tiles in flight per SM for the single DP */
    uint32_t high_levels;    /* number of tile waves = launches of the DP kernel */
    uint32_t sm_count;
} kp_plan_info;

/* Return codes.  KP_ERR_CAPACITY: the workspace `cap` the caller passed was too small for the result (kp_backtrack,
 * kp_cv_heldout, kp_dp_cv_job, kp_shard_backtrack, kp_shard_cv_heldout, kp_greedy): call again with a larger one.  Everything else is KP_ERR. */
#define KP_OK 0
#define KP_ERR 1
#define KP_ERR_CAPACITY 2

const char *kp_last_error(void);
int kp_version(void);

/* gen_pat: IUPAC general pattern, e.g. "NNNNANNNN".  device: CUDA ordinal. */
int kp_plan_create(const char *gen_pat, int device, kp_plan **out);
/* A plan WITHOUT the DP's tile lattice: digit and k-mer tables only, for the entry points that work on the k-mer tables
 * (kp_pack_counts, kp_pattern_counts, kp_greedy).  Any general pattern whose k-mer table fits the device is accepted;
 * kp_expand_counts, the DP, the backtrack and the shard functions refuse such a plan. */
int kp_plan_create_lite(const char *gen_pat, int device, kp_plan **plan);
int kp_plan_destroy(kp_plan *plan);
int kp_plan_get_info(const kp_plan *plan, kp_plan_info *out);

/*
 * K1.  h_codes[n]: one k-mer per entry, 4 bits per position (one-hot A=1,C=2,G=4,T=8), position 0 in
 * the least significant nibble; h_pos/h_neg: its positive and negative counts.  Entries naming the
 * same k-mer are summed.  d_kmerM/d_kmerU: int64[nkmer] in k-mer index order (position 0 fastest,
 * bases in the reference's `code` order).  k <= 16.
 */
int kp_pack_counts(kp_plan *plan, const uint64_t *h_codes, const int64_t *h_pos, const int64_t *h_neg, uint64_t n,
                   int64_t *d_kmerM, int64_t *d_kmerU, void *stream);

/* K2.  d_exp*: int64[expanded_elems]; counts of every (high-digit tile) x (low k-mer). */
int kp_expand_counts(kp_plan *plan, const int64_t *d_kmerM, const int64_t *d_kmerU, int64_t *d_expM,
                     int64_t *d_expU, void *stream);

/*
 * K3+K4.  Full DP.  d_best: float32[table_elems] best loss per pattern; d_kept: uint16[kept_elems], one
 * bit per pattern, set when the pattern is kept whole (its own score beat every split).  Which split won
 * is not stored: it is the first split in the reference's scan order whose float32 child sum equals the
 * minimum, and kp_backtrack / kp_split_codes re-derive it from d_best.
 * max_count: upper bound of any pattern count (n_mut + n_unmut); selects 32- or 64-bit on-chip counts.
 */
int kp_dp_single(kp_plan *plan, const int64_t *d_expM, const int64_t *d_expU, uint64_t max_count, double alpha,
                 double beta, double penalty, float *d_best, uint16_t *d_kept, void *stream);

/*
 * K5.  Optimal partition of pattern `root` (UINT64_MAX: the general pattern), dense pattern numbers in the
 * reference's emission order.  d_ws: device workspace of kp_backtrack_ws_bytes(cap).  Synchronises `stream`.
 */
uint64_t kp_backtrack_ws_bytes(uint64_t cap);
int kp_backtrack(kp_plan *plan, const float *d_best, const uint16_t *d_kept, void *d_ws, uint64_t cap, uint64_t root,
                 uint64_t *h_patnums, uint64_t *n_out, void *stream);

/*
 * The reference's backtrack pointer as a code: h_codes[i] = 0xFF if pattern h_patnums[i] is kept whole, else
 * position*8 + split_index of the winning split (bottum_up_array_w_numba.py:36-49).  Synchronises.
 */
int kp_split_codes(kp_plan *plan, const float *d_best, const uint16_t *d_kept, const uint64_t *h_patnums, uint64_t n,
                   uint8_t *h_codes, void *stream);

/* h_out[i] = table[first + i] for i < n, in dense pattern numbering (table: d_best / d_train / d_test). */
int kp_gather_table(kp_plan *plan, const float *d_table, uint64_t first, uint64_t n, float *h_out, void *stream);
/* h_out[i] = 1 if pattern first + i is kept whole. */
int kp_gather_kept(kp_plan *plan, const uint16_t *d_kept, uint64_t first, uint64_t n, uint8_t *h_out, void *stream);

/*
 * Scores (h_best), kept-whole flags (h_kept) and split codes (h_codes, as kp_split_codes) of arbitrary patterns given by
 * their dense numbers; any of the three outputs may be NULL.  Used by the full-size parity tests to pull whole
 * sub-lattices (e.g. every sub-pattern of ANNNANNNN out of the NNNNANNNN table).  Synchronises.
 */
int kp_gather_patterns(kp_plan *plan, const float *d_table, const uint16_t *d_kept, const uint64_t *h_patnums, uint64_t n,
                       float *h_best, uint8_t *h_kept, uint8_t *h_codes, void *stream);

/*
 * One cross-validation job = one fold x alpha x penalty.  d_exp?tot: all-fold totals, d_exp?test: the fold's
 * held-out counts (both from kp_expand_counts).  Train counts are total - held-out; the subtraction commutes with
 * the sums of the expansion, so the DP kernel of kp_dp_single forms them on the fly when it reads a tile's base counts
 * (no train table exists) and fills d_train (float32[table_elems]) and d_kept.  The reference additionally carries the held-out loss of every
 * pattern's best partition but only reads it at the general pattern: that number is the float32 sum, in tree
 * order, of the held-out losses of the leaves of the optimal partition, and is computed here from the
 * backtracked tree (d_ws/cap as for kp_backtrack).
 * h_top[2]: train and held-out loss of the general pattern (synchronises); NULL: DP only, no synchronisation.
 */
int kp_dp_cv_job(kp_plan *plan, const int64_t *d_expMtot, const int64_t *d_expUtot, const int64_t *d_expMtest,
                 const int64_t *d_expUtest, uint64_t max_count, double alpha, double beta_fold, double penalty,
                 float *d_train, uint16_t *d_kept, void *d_ws, uint64_t cap, float *h_top, void *stream);

/*
 * The same job without a host round trip, for callers that keep the GPU busy with the next job while this one's results
 * travel: kp_cv_job_enqueue queues the DP, the backtrack, the leaf kernel and the copies of their results into h_stage
 * (page-locked host memory of kp_cv_stage_bytes(cap) bytes) and returns without synchronising; kp_cv_job_finish, called
 * once the stream has passed that point (e.g. after an event recorded behind the call), does the host part and fills
 * h_top[2] = (train, held-out) loss of the general pattern.  d_train / d_kept must not be overwritten before the
 * stream has passed the enqueue (two tables in rotation suffice: work on one stream runs in order).
 */
uint64_t kp_cv_stage_bytes(uint64_t cap);
int kp_cv_job_enqueue(kp_plan *plan, const int64_t *d_expMtot, const int64_t *d_expUtot, const int64_t *d_expMtest,
                      const int64_t *d_expUtest, uint64_t max_count, double alpha, double beta_fold, double penalty,
                      float *d_train, uint16_t *d_kept, void *d_ws, uint64_t cap, void *h_stage, void *stream);
int kp_cv_job_finish(const void *h_stage, uint64_t cap, float *h_top);

/*
 * Held-out loss of the best partition of pattern `root` after kp_dp_cv_job (the reference's test_score_mem[root],
 * bottum_up_array_penalty_plus_pseudo_CV.py:46-51, :71-78), same total / held-out tables as the job.  Synchronises.
 */
int kp_cv_heldout(kp_plan *plan, const float *d_train, const uint16_t *d_kept, const int64_t *d_expMtot,
                  const int64_t *d_expUtot, const int64_t *d_expMtest, const int64_t *d_expUtest, double alpha,
                  double beta_fold, double penalty, uint64_t root, void *d_ws, uint64_t cap, float *h_test, void *stream);

/* Counts of arbitrary patterns (dense numbers) straight from the k-mer tables.  Synchronises. */
int kp_pattern_counts(kp_plan *plan, const int64_t *d_kmerM, const int64_t *d_kmerU, const uint64_t *h_patnums,
                      uint64_t n, int64_t *h_M, int64_t *h_U, void *stream);

/*
 * Scoring a fitted partition on k-mer counts (replaces the reference's papa.PatternPartition check, papa.py:53-107, and
 * its get_loss on new data).  h_patnums[n]: the partition's patterns as dense pattern numbers of the plan's general
 * pattern, in file order (1 <= n < 2^32 - 1).  Any plan works; a lite plan is enough.
 *
 * kp_partition_assign fills d_owner (uint32[nkmer]) with the index of the pattern that covers each k-mer
 * (0xFFFFFFFF: none) and reports *h_conflict = 1 + the smallest k-mer index covered twice and *h_uncovered = 1 + the
 * smallest k-mer index covered by no pattern, each 0 when there is none.  Members of the patterns are claimed in
 * file order in chunks of nkmer; the first chunk that finds a k-mer claimed twice ends the pass, so *h_conflict is the
 * smallest k-mer covered twice within the chunks up to it (all of them when the sizes sum to at most nkmer), and
 * *h_uncovered is 0 then.  At most two chunks run.  Synchronises.
 *
 * kp_partition_score: per pattern, the counts M[q], U[q] of its k-mers in d_kmerM / d_kmerU (kp_pack_counts layout)
 * and h_t[q] = xlogy(M, p) + xlog1py(U, -p) in float64 with p = h_rate[q] (bit for bit as scipy evaluates it).  Refused
 * when the pattern sizes sum to more than nkmer.  d_kmer_rate (optional, double[nkmer]): the rate of each k-mer's
 * owner in d_owner from kp_partition_assign (NaN where there is none).  Synchronises.  Every output is the same on
 * every run.
 */
int kp_partition_assign(kp_plan *plan, const uint64_t *h_patnums, uint64_t n, uint32_t *d_owner, uint64_t *h_conflict,
                        uint64_t *h_uncovered, void *stream);
int kp_partition_score(kp_plan *plan, const uint64_t *h_patnums, const double *h_rate, uint64_t n, const int64_t *d_kmerM,
                       const int64_t *d_kmerU, const uint32_t *d_owner, double *d_kmer_rate, int64_t *h_M, int64_t *h_U,
                       double *h_t, void *stream);

/* Applying a partition along sequences (DESIGN §4c; kmerpapa_b200/apply_partition.py).  Position i of a record of
 * length rec_len has the window seq[i - c, i - c + k), c = k / 2.  The window is a context when it lies in the record
 * and all its bytes are A, C, G or T (either case).  It matches when every base lies in the general pattern's letter at
 * its position; its k-mer index is kp_pack_counts'.  With both != 0 (odd k only) the reverse complement of the window is
 * looked up too, and the position's rate is p_fwd + p_rev (one float64 addition; a side that does not match adds 0).
 *
 * kp_kmer_rates: d_kmer_rate (double[nkmer]) = h_rate of each k-mer's owner in d_owner from kp_partition_assign (NaN
 * where there is none).  Synchronises.
 *
 * kp_seq_scan: one pass over the positions [pos0, pos1) of a record; pos0 is a multiple of the piece size 65536.
 * d_seq holds the record bytes [seq_base, seq_base + seq_len), 16-byte aligned and readable up to the next multiple of
 * 16 bytes; it must hold every window of the positions that lies in the record.  Without d_tasks, block b sums piece
 * pos0 / 65536 + b of the record (its positions in [pos0, pos1)): d_sum[b] = its float64 rate sum by a fixed tree and
 * d_n[b] = its matching (position, strand) pairs.  Optionally d_track[i - pos0] = RN_f32(rate of position i), NaN where i
 * has no context; and d_counts[kidx] (int64[nkmer], not zeroed here) += 1 per match of a position i whose bit
 * i - pos0 is set in d_count_mask (uint32 words; NULL: every position).  With d_tasks (uint32[ntask][3]: piece of the
 * record, lo, hi), entry t gives in d_sum[t], d_n[t] the same sums restricted to positions piece * 65536 + [lo, hi),
 * through the same tree with zeros elsewhere: where a task covers the whole piece its sum is the piece's sum, bit for
 * bit; tracks and counts are refused there.  Does not synchronise.
 *
 * kp_region_sums: for region r = d_regions[4r..4r+3] = (first piece pa, last piece pb, task of pa or -1, task of pb or
 * -1), d_sum[r] / d_n[r] = the left-to-right float64 / int64 sums over the pieces pa..pb of the task sums d_task_sum /
 * d_task_n where a task is given and of the piece sums d_piece_sum / d_piece_n elsewhere.  Does not synchronise.
 * Every output is the same on every run and for every split of a record into calls. */
int kp_kmer_rates(kp_plan *plan, const uint32_t *d_owner, const double *h_rate, uint64_t n, double *d_kmer_rate, void *stream);
int kp_seq_scan(kp_plan *plan, const uint8_t *d_seq, uint64_t seq_base, uint64_t seq_len, uint64_t rec_len, uint64_t pos0,
                uint64_t pos1, int both, const double *d_kmer_rate, const uint32_t *d_tasks, uint64_t ntask, double *d_sum,
                int64_t *d_n, float *d_track, const uint32_t *d_count_mask, int64_t *d_counts, void *stream);
int kp_region_sums(kp_plan *plan, const double *d_piece_sum, const int64_t *d_piece_n, const double *d_task_sum,
                   const int64_t *d_task_n, const int64_t *d_regions, uint64_t n, double *d_sum, int64_t *d_n, void *stream);

/* Counting the contexts of SNVs (DESIGN §4d; kmerpapa_b200/count_mutations.py), with the windows, matching and k-mer
 * index of kp_seq_scan.  d_seq, seq_base, seq_len, rec_len, pos0, pos1 and both are as in kp_seq_scan, except that pos0
 * need not be a multiple of 65536 and d_seq need not be aligned.  SNV t is at record position d_pos[t] (int64, in
 * [pos0, pos1)) with d_ref_alt[t] = REF code | ALT code << 2 (A, C, G, T = 0..3).  d_status[t] gets the first that
 * applies of:
 *   KP_SNV_REF_MISMATCH     the genome byte is a base (either case) other than REF;
 *   KP_SNV_OUTSIDE_REGIONS  bit pos - pos0 of d_count_mask (uint32 words; NULL: every position) is clear;
 *   KP_SNV_NO_CONTEXT       the window leaves the record or holds a byte that is not a base;
 *   KP_SNV_NO_MATCH         neither the forward window nor (both != 0) the reverse one matches;
 *   KP_SNV_ALT_NOT_SELECTED alt_slot[a] < 0, where a is ALT when the forward window matches, else complement(ALT);
 *   KP_SNV_COUNTED          d_counts[alt_slot[a] * nkmer + kidx] += 1 (int64, not zeroed here), with kidx the index of
 *                           the forward window when it matches, else of the reverse one.
 * A d_pos outside [pos0, pos1) gets KP_SNV_BAD_POSITION and touches nothing else.  alt_slot: 4 host ints, each -1..3.
 * The counts are integer atomics, so they are the same whatever the thread order and the split into calls.  Does not
 * synchronise. */
#define KP_SNV_REF_MISMATCH 0
#define KP_SNV_OUTSIDE_REGIONS 1
#define KP_SNV_NO_CONTEXT 2
#define KP_SNV_NO_MATCH 3
#define KP_SNV_ALT_NOT_SELECTED 4
#define KP_SNV_COUNTED 5
#define KP_SNV_BAD_POSITION 255
int kp_snv_counts(kp_plan *plan, const uint8_t *d_seq, uint64_t seq_base, uint64_t seq_len, uint64_t rec_len, uint64_t pos0,
                  uint64_t pos1, int both, const int64_t *d_pos, const uint8_t *d_ref_alt, uint64_t n, const int *alt_slot,
                  const uint32_t *d_count_mask, int64_t *d_counts, uint8_t *d_status, void *stream);

/* Counting the SNVs of several models per region (DESIGN §4e; kmerpapa_b200/burden.py).  The n SNVs of one record are
 * at d_pos (int64, sorted ascending) and d_model[t] (uint8) is the model that counts SNV t; an id >= nmodels (255: none)
 * counts for no model.  nmodels is 1..255.  For region r = d_regions[2r..2r+1] = (start, end), half-open in the
 * coordinates of d_pos, d_observed[r * nmodels + m] (int64) = the SNVs t with start <= d_pos[t] < end and d_model[t] = m.
 * Regions may overlap and come in any order; one with end <= start counts nothing.  A per-model prefix count over the
 * SNVs (a three-pass block scan) makes each region cost two binary searches and nmodels differences, whatever its
 * length.  d_ws: device workspace of kp_snv_region_ws_bytes(n, nmodels) bytes; d_pos, d_regions, d_ws and d_observed
 * are 8-byte aligned.  The counts are integers, the same on every run.  Does not synchronise. */
uint64_t kp_snv_region_ws_bytes(uint64_t n, int nmodels);
int kp_snv_region_counts(kp_plan *plan, const int64_t *d_pos, const uint8_t *d_model, uint64_t n, int nmodels,
                         const int64_t *d_regions, uint64_t nreg, void *d_ws, int64_t *d_observed, void *stream);

/* Where a dense pattern number lives in the device layout: element of a float table, element and bit of d_kept. */
int kp_pattern_offset(const kp_plan *plan, uint64_t patnum, uint64_t *table_elem, uint64_t *kept_elem, uint32_t *kept_bit);

/* Number of kernel launches issued through this plan so far (for bench.py's gpu_launches). */
uint64_t kp_plan_launch_count(const kp_plan *plan);
/* Name of the kernel family kp_dp_single / kp_dp_cv_job launch for this plan at one count width (reports, bench.py's
 * roofline.kernel): wide = 0 for a max_count of at most 2^32 - 1 (32-bit on-chip counts), wide != 0 above.  The fiber
 * kernel needs more shared memory for 64-bit counts, so the two widths can run different families. */
const char *kp_dp_kernel_name(const kp_plan *plan, int wide);

/* ---------------------------------------------------------------------------------------------------
 * One DP sharded over the GPUs of a node (SURVEY 8f.3: pattern-space sharding; the reference has no
 * counterpart, its tables are single numpy arrays, bottum_up_array_w_numba.py:82-91).
 *
 * The score table is split by the digit of the TOP high position of the tile number; every rank (one process per
 * GPU, or several shards in one process) owns the tiles of its digits and runs the same waves on them.  The
 * children of a tile along the top position may live on a peer: the DP kernel loads them from the peer's memory
 * (NVLink) in the same pipeline as the local ones.  The caller synchronises the ranks between waves
 * (torch.distributed barrier / all_reduce on the same stream) and provides every rank with the FULL expanded
 * count tables (kp_expand_counts is cheap and replicated).
 *
 *   kp_shard_create -> exchange pointers (kp_ipc_export / all_gather / kp_ipc_open, or directly within one
 *   process) -> kp_shard_set_peer for every other rank -> for wave in 0..nwaves-1: kp_shard_dp_wave, barrier ->
 *   kp_shard_backtrack / kp_shard_gather on any rank.  A cross-validation job: kp_shard_cv_wave instead of
 *   kp_shard_dp_wave, then kp_shard_cv_heldout on any rank.
 * ------------------------------------------------------------------------------------------------- */
typedef struct kp_shard kp_shard;

typedef struct kp_shard_info {
    uint64_t local_tiles;   /* tiles stored on this rank */
    uint64_t table_elems;   /* float32 elements of this rank's score shard */
    uint64_t kept_elems;    /* uint16 elements of this rank's kept-whole shard */
    uint64_t d_best;        /* device pointer of the score shard (cudaMalloc: exportable with kp_ipc_export) */
    uint64_t d_kept;        /* device pointer of the kept-whole shard */
    uint32_t rank, world;
    uint32_t nwaves;        /* waves of the DP (the same on every rank) */
    uint32_t top_digits;    /* digits of the top high position owned by this rank */
    uint32_t replicate;     /* 1: replicated mode */
    uint32_t reserved;
} kp_shard_info;

/* owner rank and local slot of every digit of the top high position (16 entries each) for `world` ranks */
int kp_shard_assignment(const kp_plan *plan, int world, uint8_t *owner16, uint8_t *slot16);
/* allocate this rank's shard on the plan's device; world <= min(8, radix of the top position); needs an N position.
 * replicate = 0 (capacity): a rank stores only its own tiles and the kernel LOADS peer children over NVLink;
 * replicate = 1 (speed): every rank allocates a full-size table, the kernel reads locally and PUSHES each finished
 *   row into the table of every peer that owns a superset digit (posted NVLink writes). */
int kp_shard_create(kp_plan *plan, int rank, int world, int replicate, kp_shard **out);
int kp_shard_destroy(kp_shard *shard);
int kp_shard_get_info(const kp_shard *shard, kp_shard_info *out);
/* device pointers (valid on this rank's device: peer-mapped) of rank `peer`'s shard */
int kp_shard_set_peer(kp_shard *shard, int peer, const float *d_best, const uint16_t *d_kept);
/* CUDA IPC plumbing: 64-byte handle of a cudaMalloc allocation; map / unmap a peer's allocation on `device` */
int kp_ipc_export(const void *d_ptr, uint8_t *handle64);
int kp_ipc_open(int device, const uint8_t *handle64, void **d_ptr);
int kp_ipc_close(int device, void *d_ptr);
/* this rank's tiles of one wave (same arguments as kp_dp_single; d_expM/d_expU are the full expanded tables).
 * All ranks must have finished wave w-1 before any rank starts wave w. */
int kp_shard_dp_wave(kp_shard *shard, int wave, const int64_t *d_expM, const int64_t *d_expU, uint64_t max_count,
                     double alpha, double beta, double penalty, void *stream);
/* kp_shard_dp_wave on train counts d_exp?tot - d_exp?test (one CV job, one wave); same rules as kp_shard_dp_wave */
int kp_shard_cv_wave(kp_shard *shard, int wave, const int64_t *d_expMtot, const int64_t *d_expUtot,
                     const int64_t *d_expMtest, const int64_t *d_expUtest, uint64_t max_count,
                     double alpha, double beta_fold, double penalty, void *stream);
/* after the last kp_shard_cv_wave on every rank: h_top[0] = train loss of `root`, h_top[1] = held-out loss of the
 * best partition of `root` (kp_cv_heldout's definition), read through the shard view.  Synchronises. */
int kp_shard_cv_heldout(kp_shard *shard, const int64_t *d_expMtot, const int64_t *d_expUtot, const int64_t *d_expMtest,
                        const int64_t *d_expUtest, double alpha, double beta_fold, double penalty, uint64_t root,
                        void *d_ws, uint64_t cap, float *h_top, void *stream);
/* like kp_backtrack, over all shards (reads peers' memory); callable on any rank after the last wave */
int kp_shard_backtrack(kp_shard *shard, void *d_ws, uint64_t cap, uint64_t root, uint64_t *h_patnums, uint64_t *n_out,
                       void *stream);
/* score / kept-whole flag / split code (any of the outputs may be NULL) of arbitrary patterns, from any shard */
int kp_shard_gather(kp_shard *shard, const uint64_t *h_patnums, uint64_t n, float *h_best, uint8_t *h_kept,
                    uint8_t *h_codes, void *stream);

/* Greedy top-down partition (reference: greedy_penalty_plus_pseudo.py:155-196 greedy_res_kmer_table_ord, :285-300
 * greedy_partition, :318-337 CrossValidation.loglik).  Starting from the general pattern, a pattern is split at the
 * first (string position, split) whose float64 sum of the two children's losses is the strict minimum below the
 * pattern's own loss, else it becomes a leaf; children are expanded first child first.  Works on the dense k-mer
 * tables of kp_pack_counts (no pattern table).  d_testM/d_testU (both or none): held-out k-mer tables; h_test then
 * receives the held-out -2 log-likelihood of every leaf under the leaf's train rate (test_logLik, :26-34).
 * Outputs: dense pattern numbers of the leaves in the reference's order, their float64 losses, and h_total = the
 * float64 sum of the losses in the order of the recursion (the reference's returned score). */
uint64_t kp_greedy_ws_bytes(uint64_t cap);
int kp_greedy(kp_plan *plan, const int64_t *d_kmerM, const int64_t *d_kmerU, const int64_t *d_testM, const int64_t *d_testU,
              double alpha, double beta, double penalty, void *d_ws, uint64_t cap, uint64_t *h_patnums, double *h_loss,
              double *h_test, uint64_t *n_out, double *h_total, void *stream);

/* The all-k-mers model (reference: all_kmers_CV.py:8-13, :42-43; `--score all_kmers`): for n (k-mer, fold) items with
 * train counts (Mtr, Utr), held-out counts (Mte, Ute) and the fold's beta, the float64 terms
 *   train = -2 (xlogy(Mtr, p) + xlog1py(Utr, -p)),  test = -2 (xlogy(Mte, p) + xlog1py(Ute, -p)),
 *   p = (Mtr + alpha) / (Mtr + Utr + alpha + beta), bit for bit as numpy/scipy evaluate them.  Host buffers. */
int kp_kmer_fold_terms(int device, const int64_t *h_Mtr, const int64_t *h_Utr, const int64_t *h_Mte, const int64_t *h_Ute,
                       const double *h_beta, uint64_t n, double alpha, double *h_train, double *h_test);

/* Test hook: y[i] = device log(x[i]) (the glibc-exact restatement used by the scoring kernels). */
int kp_debug_log(int device, const double *h_x, double *h_y, uint64_t n);
/* Test hook: level-0 score of (M,U) pairs on the device (scipy xlogy/xlog1py restated). */
int kp_debug_leaf_score(int device, const int64_t *h_M, const int64_t *h_U, uint64_t n, double alpha, double beta,
                        double penalty, double *h_out);
/* Test hook: the three level >= 1 scoring paths of the DP kernels, item by item.  Item i has the per-base counts
 * h_M[4i..4i+3], h_U[4i..4i+3] (>= 0; the pattern's counts are their sums), its own alpha, beta and penalty, and
 * h_wide[i] = 1 for 64-bit on-chip counts, 0 for 32-bit (refused when the counts sum to 2^32 or more).  Outputs:
 * h_lb = the score filter's float32 lower bound; h_ok, h_sf, h_rup, h_fast = kp_self_score_fast's verdict,
 * RN_f32(s), "rounded up" bit and float64 estimate s~; h_exact = the exact float64 score.  Host buffers. */
int kp_debug_self_score(int device, const int64_t *h_M, const int64_t *h_U, const double *h_alpha, const double *h_beta,
                        const double *h_penalty, const uint8_t *h_wide, uint64_t n, float *h_lb, uint8_t *h_ok, float *h_sf,
                        uint8_t *h_rup, double *h_fast, double *h_exact);

#ifdef __cplusplus
}
#endif
#endif /* KMERPAPA_B200_H */
