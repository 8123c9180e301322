/*
 * basevar_b200.h -- C ABI of the B200-native `basevar basetype` per-site statistical core.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference has no FFI layer; the seam
 * it exposes is the C++ class `BaseType` and the free function `strand_bias`:
 *
 *   reference interface                                         replaced by
 *   ----------------------------------------------------------  ---------------------------------
 *   struct BatchInfo                    src/basetype.h:25-43     bv_tile (packed SoA planes), or bv_sparse_tile: the
 *                                                                covered cells only, expanded on the device
 *   BaseType::BaseType(BatchInfo*,af)   src/basetype.h:105       bv_tile_submit / bv_tile_submit_sparse / bv_tile_run_device
 *                                       src/basetype.cpp:22-72   (count kernel: depths, strand table)
 *   BaseType::lrt()                     src/basetype.h:117-118   same call (scalar / bound / EM kernels)
 *                                       src/basetype.cpp:130-199
 *   EM / e_step / m_step                src/algorithm.h:148-255  same call
 *   chi2_test -> kf_gammaq              src/algorithm.h:44-46    same call
 *   strand_bias(...)                    src/basetype.h:178-181   same call (fwd/rev counts + FS)
 *                                       src/basetype.cpp:244-295
 *   fisher_exact_test -> kt_fisher_exact src/algorithm.h:62-74   same call; bv_fisher_fs for a free-standing 2x2 table
 *   getters get_alt_bases/get_lrt_af/   src/basetype.h:120-151   fields of bv_site_out
 *     get_var_qual/get_total_depth/get_base_depth
 *   per-site driver _basevar_caller     src/basetype_caller.cpp:667-765   caller loops over bv_site_out
 *   ref_vs_alt_ranksumtest(...) x3      src/basetype.h:168-176   bv_tile_submit_calls (rank-sum kernel), bv_call_out
 *     (MQRankSum/ReadPosRankSum/BaseQRankSum of the VCF row, src/basetype_caller.cpp:1151-1157)
 *   __gb(): BaseType on one population  src/basetype_caller.cpp:767-797   bv_set_groups + bv_tile_submit_calls
 *     group + lrt([REF, ALT...])        src/basetype_caller.cpp:747-760   (group kernel), bv_group_out
 *   BaseType::lrt(specific_bases)       src/basetype.h:118               bv_tile_submit_lists / bv_tile_run_device_lists
 *     (any ordered candidate list)      src/basetype.cpp:130-199         (list kernel K8), bv_lrt_out
 *   ref_vs_alt_ranksumtest(...) for any src/basetype.h:168-176           bv_ranksum_test (rank-sum test kernel K9), one double
 *     ALT set and value list            src/basetype.cpp:201-242         per free-standing problem
 *   the VCF row of a tile in batch:     src/basetype_caller.cpp:1151-1194 bv_tile_submit_sparse_calls / bv_tile_submit_calls with
 *     rank sums + groups, compact form                                    BV_OUT_COMPACT, bv_tile_wait_calls_compact
 *   lrt([REF, ALT...]) at called sites  src/basetype_caller.cpp:747-760   bv_tile_submit_sparse_lists (K8 on the expanded planes);
 *     of a sparse tile                                                    with BV_OUT_COMPACT one packed entry per listed site,
 *                                                                         bv_tile_wait_lists_compact
 *
 * Everything is `extern "C"`, plain pointers and sizes, POD structs; no exception crosses the
 * boundary.  Every entry point returns BV_OK (0) or a negative status; bv_last_error() gives text.
 * A context is bound to one CUDA device and must not be shared between host threads; use one
 * context per (GPU, host worker).  Calls on one slot are stream ordered.
 *
 * There is NO CPU fallback: without a usable CUDA device bv_create() fails with BV_ERR_CUDA.
 */
#ifndef BASEVAR_B200_H
#define BASEVAR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BV_VERSION_MAJOR 0
#define BV_VERSION_MINOR 1

/* ---- status codes ---------------------------------------------------------------------------- */
#define BV_OK            0
#define BV_ERR_ARG      -1   /* bad argument (null pointer, pitch not multiple of 16, tile too large) */
#define BV_ERR_CUDA     -2   /* CUDA runtime error or no device; text in bv_last_error()            */
#define BV_ERR_STATE    -3   /* slot busy / nothing submitted                                         */
#define BV_ERR_NOMEM    -4

/* ---- cell encoding of the packed SoA planes (one u8 per sample per site, per plane) ---------- */
/* base plane: first character of BatchInfo::align_bases[i] (src/basetype.cpp:50)                  */
#define BV_BASE_A      0
#define BV_BASE_C      1
#define BV_BASE_G      2
#define BV_BASE_T      3
#define BV_BASE_OTHER  4   /* any other single character: counted in total depth, never an allele    */
                           /* (src/basetype.cpp:58-64 gives it the row {e/3,e/3,e/3,e/3})            */
#define BV_BASE_N      5   /* 'N' = uncovered / masked: skipped (src/basetype.cpp:51)                 */
#define BV_BASE_INS    6   /* "+SEQ": skipped by the SNP caller                                       */
#define BV_BASE_DEL    7   /* "-SEQ": skipped by the SNP caller                                       */
/* qual plane: phred = align_base_quals[i] - 33, 0..93 (src/basetype.cpp:47)                        */
#define BV_QUAL_MAX    93
/* strand plane: map_strands[i] */
#define BV_STRAND_FWD  0   /* '+' */
#define BV_STRAND_REV  1   /* '-' */
#define BV_STRAND_NONE 2   /* '.' (uncovered) or '*' */

/* ---- per-site flags --------------------------------------------------------------------------- */
#define BV_FLAG_BAD_STRAND   0x01u /* counted cell whose strand is not +/-: reference throws (basetype.cpp:271) */
#define BV_FLAG_BAD_QUAL     0x02u /* counted cell with phred > 93, at a site whose result depends on qualities  */
#define BV_FLAG_ZERO_SUBSET  0x04u /* a candidate subset has zero depth: reference throws (basetype.cpp:113)  */
#define BV_FLAG_MONO_QUAL    0x08u /* QUAL came from the mono-allelic 5000 rule (basetype.cpp:182-185)        */
#define BV_FLAG_NEAR_LRT     0x10u /* some LRT decision had |chi2 - threshold| < 1e-9*threshold (possible flip) */
#define BV_FLAG_LRT_BOUND    0x20u /* the LRT outcome (drop the minor allele) was proven by a bound, no EM ran:   */
                                   /* chi2 and em_calls of the record are 0 (the reference exposes neither here)  */
#define BV_FLAG_EM_MAXITER   0x40u /* an EM used all em_max_iter iterations                                   */
#define BV_FLAG_LRT_TIE      0x80u /* two candidate subsets had equal chi2 (to rounding): first one kept       */

#define BV_EM_ABS_INT_TRUNC 0  /* as built by g++/glibc: abs() resolves to int abs(int) (algorithm.h:245)   */
#define BV_EM_ABS_DOUBLE    1  /* fabs(): the evident intent                                                */

#define BV_LOC_HOST   0
#define BV_LOC_DEVICE 1

/* ---- parameters ------------------------------------------------------------------------------- */
typedef struct bv_params {
    float    min_af;         /* CLI --min-af as FLOAT (basetype_utils.h:80), widened to double inside;    */
                             /* caller applies min(100.0f/n_bam, min_af) (basetype_caller.cpp:122)        */
    int32_t  lrt_threshold;  /* 24  (basetype.h:21)                                                       */
    int32_t  em_max_iter;    /* 100 (algorithm.h:213)                                                     */
    float    em_eps;         /* 0.001f (algorithm.h:213)                                                  */
    int32_t  em_abs_mode;    /* BV_EM_ABS_*                                                               */
    uint32_t max_samples;    /* capacity: largest n_samples of any tile                                   */
    uint32_t max_sites;      /* capacity: largest n_sites of any tile submitted through a slot            */
    uint32_t n_slots;        /* in-flight tile slots (each owns a stream + pinned staging); >= 1          */
    uint32_t reserved;
} bv_params;

/* ---- one tile of the packed site-major SoA pileup --------------------------------------------- */
typedef struct bv_tile {
    const uint8_t* base;     /* [n_sites][pitch]  BV_BASE_*                                               */
    const uint8_t* qual;     /* [n_sites][pitch]  phred                                                   */
    const uint8_t* strand;   /* [n_sites][pitch]  BV_STRAND_*                                             */
    const uint8_t* ref_base; /* [n_sites] raw ASCII of BatchInfo::ref_base[0] (may be lowercase or 'N')  */
    uint64_t pitch;          /* bytes between consecutive site rows, multiple of 16, >= n_samples;        */
                             /* padding cells [n_samples, pitch) are ignored                              */
    uint32_t n_sites;
    uint32_t n_samples;
    int32_t  location;       /* BV_LOC_HOST (pinned or pageable) or BV_LOC_DEVICE                         */
    int32_t  out_mode;       /* BV_OUT_RECORDS, or BV_OUT_COMPACT (host tiles; collect with bv_tile_wait_compact) */
} bv_tile;
/* Device-resident tiles have no compact form.  bv_tile_submit_calls (device tile), bv_tile_run_device_calls and
 * bv_tile_run_device_lists refuse out_mode BV_OUT_COMPACT with BV_ERR_ARG; bv_tile_run_device, and bv_tile_submit of a device
 * tile, do not read out_mode and return records. */

/* ---- per-site result record: fixed 128 bytes --------------------------------------------------- */
typedef struct bv_site_out {
    uint32_t depth[4];       /* A,C,G,T read counts       (BaseType::get_base_depth)                      */
    uint32_t depth_other;    /* BV_BASE_OTHER cells; total depth = sum(depth)+depth_other                 */
    uint32_t reserved0;      /* 0                                                                         */
    uint32_t fwd[4];         /* '+' strand count per base (strand_bias, any ALT set derivable on host)    */
    uint32_t rev[4];         /* '-' strand count per base                                                 */
    uint8_t  n_alt;          /* number of ALT alleles (0 => not a variant site)                           */
    uint8_t  alt[4];         /* ALT base codes, in the reference's order (ACGT order of the active set)   */
    uint8_t  n_active;       /* |active_bases| after backward elimination                                 */
    uint8_t  flags;          /* BV_FLAG_*                                                                 */
    uint8_t  em_calls;       /* number of EM invocations (saturating)                                     */
    double   af[4];          /* AF by EM+LRT for alt[i] (BaseType::get_lrt_af); may be NaN (Q0 read)      */
    double   qual;           /* BaseType::get_var_qual(); 0 when n_alt == 0                               */
    double   chi2;           /* last chi_sqrt_value of the LRT loop (0 when the loop did not run)         */
    double   fs_cvg;         /* FS of strand_bias(ref, all non-ref ACGT): the CVG row (caller.cpp:1245)   */
    double   fs_vcf;         /* FS of strand_bias(ref, ALT set): the VCF row (caller.cpp:1164); 0 if !n_alt */
} bv_site_out;

/* ---- compact record transport ---------------------------------------------------------------------
 * At < 1x nine sites in ten show nothing but the reference base (or nothing at all): their whole 128-byte record follows
 * from two counts.  With BV_OUT_COMPACT a tile returns 8 bytes for every site and a full record only for the others (~12 %
 * at 0.1x): 24 bytes per site instead of 128 across PCIe and through the host's memory.
 *   w0 bit 31 clear: every counted read shows REF: w0 = depth[REF], w1 = how many of them are on the '-' strand (both 0
 *                    when no read is counted, or REF is not A/C/G/T); bv_site_expand() rebuilds the record;
 *   w0 bit 31 set:   w0 & 0x7fffffff = index of the site's record in the tile's list of full records. */
#define BV_OUT_RECORDS 0
#define BV_OUT_COMPACT 1
typedef struct bv_site_brief {
    uint32_t w0;
    uint32_t w1;
} bv_site_brief;

/* ---- synthetic pileup model (bench / tests); integer thresholds only, so that the device       */
/* generator and its host twin are bit-identical                                                   */
typedef struct bv_synth_model {
    uint64_t seed;
    uint32_t cov_thr;        /* cell covered iff u32 draw < cov_thr                                       */
    uint32_t var_thr;        /* site is variant iff u32 draw < var_thr                                    */
    uint32_t multi_thr;      /* variant site gets extra ALT alleles iff u32 draw < multi_thr              */
    uint32_t q_lo;           /* phred = q_lo + ((u32 draw * q_span) >> 32)                                */
    uint32_t q_span;
    uint32_t reserved;
    uint32_t err_thr[96];    /* per phred: read is an error iff 24-bit draw < err_thr[q]                  */
    uint32_t af_thr[1024];   /* inverse CDF of the ALT1 allele frequency as a u32 threshold               */
    uint32_t af_extra_thr[256]; /* same for ALT2/ALT3 of multi-allelic sites                              */
} bv_synth_model;

/* ---- called sites (n_alt > 0): the extra inputs and outputs of the VCF row ------------------------ */
/* Planes the reference reads only at called sites (src/basetype_caller.cpp:1151-1157).  Same site-major layout as
 * bv_tile; rows are fetched for the called sites only, so pinned host planes are read in place over PCIe. */
typedef struct bv_tile_aux {
    const uint8_t*  mapq;    /* [n_sites][pitch]      BatchInfo::mapqs, 0..255 (same pitch as the tile)             */
    const uint16_t* rpr;     /* [n_sites][rpr_pitch]  BatchInfo::base_pos_ranks (read position rank), 0..65535      */
    uint64_t rpr_pitch;      /* ELEMENTS between consecutive rows of `rpr`, multiple of 8, >= n_samples             */
} bv_tile_aux;

/* One per site with n_alt > 0, in NO particular order (`site` identifies the row).  16 bytes.
 * Each rank sum is (int) ref_vs_alt_ranksumtest(upper REF, ALT string, first bases, values): the phred-scaled
 * two-sided Wilcoxon p of REF reads vs reads of the called ALT alleles, 10000 when either class is empty or p == 0
 * (src/basetype.cpp:201-242, src/algorithm.h:76-136), truncated to int as src/basetype_caller.cpp:1151-1157 does. */
typedef struct bv_call_out {
    uint32_t site;               /* row index inside the tile                        */
    int32_t  mq_rank_sum;        /* values = mapqs                                   */
    int32_t  read_pos_rank_sum;  /* values = base_pos_ranks                          */
    int32_t  base_q_rank_sum;    /* values = align_base_quals                        */
} bv_call_out;

/* One per (called site, population group): BaseType over the group's samples + lrt([upper REF, ALT...])
 * (src/basetype_caller.cpp:747-760,767-797).  n_alt == 0: the group reports no AF (no "<group>_AF=" entry,
 * src/basetype_caller.cpp:1184-1194).  40 bytes. */
typedef struct bv_group_out {
    uint8_t n_alt;
    uint8_t alt[4];          /* base codes, in the order of the group's BaseType::get_alt_bases()                  */
    uint8_t flags;           /* BV_FLAG_* raised by the group's EM / LRT                                           */
    uint8_t reserved[2];
    double  af[4];           /* get_lrt_af(alt[i])                                                                 */
} bv_group_out;

#define BV_GROUP_NONE 255    /* sample belongs to no population group */
#define BV_MAX_GROUPS 254

/* One per site of a lists submit: BaseType(row, min_af) + lrt(list) over that site's ordered candidate list
 * (src/basetype.h:117-118, src/basetype.cpp:130-199).  64 bytes.
 *   active  = the list entries with depth/total >= min_af, in LIST order (total includes depth_other; 0 => none);
 *   EM + backward elimination over `active`, subsets in list order (src/external/combinations.h), first minimum kept;
 *   ALT     = active bases, in list order, that are not toupper(REF); af[k] = get_lrt_af(alt[k]);
 *   qual    = get_var_qual(): 5000 (BV_FLAG_MONO_QUAL) for one active base at total > 10 and depth/total > 0.5,
 *             else -10 log10 of the chi-square survival function of `chi2`; 0 when n_alt == 0;
 *   fs      = FS of strand_bias(REF, ALT set) from the record's strand table, as bv_fisher_fs computes it; 0 if !n_alt.
 * flags: BV_FLAG_ZERO_SUBSET / NEAR_LRT / LRT_TIE / EM_MAXITER / MONO_QUAL of this call, plus the row's BAD_QUAL and
 * BAD_STRAND.  A site with an empty list, or without counted reads, gets an all-zero entry.
 * Departure from the reference (which does not define the case): a list with a repeated base or a code outside
 * BV_BASE_A..BV_BASE_T is refused with BV_ERR_ARG by bv_tile_submit_lists. */
typedef struct bv_lrt_out {
    uint8_t n_alt;
    uint8_t alt[4];          /* base codes, in list order                                                          */
    uint8_t n_active;        /* |active set| after backward elimination                                            */
    uint8_t flags;           /* BV_FLAG_*                                                                          */
    uint8_t em_calls;        /* EM invocations of this call (saturating)                                           */
    double  af[4];
    double  qual;
    double  chi2;            /* last chi_sqrt_value of the elimination loop (0 when it did not run)                 */
    double  fs;
} bv_lrt_out;

/* lists[site][4]: 1..4 distinct base codes in caller order, ended early by BV_LIST_END (an empty list skips the site) */
#define BV_LIST_END 255

typedef struct bv_ctx bv_ctx;

/* ---- lifecycle --------------------------------------------------------------------------------- */
int         bv_version(void);                                  /* major*1000 + minor */
int         bv_create(int device, const bv_params* params, bv_ctx** out_ctx);
void        bv_destroy(bv_ctx* ctx);
const char* bv_last_error(const bv_ctx* ctx);                  /* ctx may be NULL: last global error */
int         bv_set_params(bv_ctx* ctx, const bv_params* params); /* change min_af / em mode; capacities fixed */
uint64_t    bv_launch_count(const bv_ctx* ctx);                /* kernels launched by this context so far */
uint64_t    bv_h2d_bytes(const bv_ctx* ctx);                   /* bytes uploaded by the bv_tile_submit* calls so far: the planes
                                                                  or cells of host tiles, and the lists of lists tiles */
/* Instrumentation: with profiling on, every tile records CUDA events between its kernels (K1 count, K2 scalar,
 * K3 bound, K4 = K4a row histograms + K4b EM tasks and decisions, then the Fisher tests K2 and K4b listed);
 * bv_last_kernel_times() waits for the most recent tile and returns the durations of K1..K4 in ms,
 * bv_last_em_kernel_times() those of K4a and K4b, bv_last_fisher_kernel_time() that of bv_fisher_kernel. */
int         bv_set_profiling(bv_ctx* ctx, int on);
int         bv_last_kernel_times(bv_ctx* ctx, float ms[4]);
int         bv_last_em_kernel_times(bv_ctx* ctx, float ms[2]);
int         bv_last_fisher_kernel_time(bv_ctx* ctx, float* ms);
int         bv_last_call_kernel_times(bv_ctx* ctx, float ms[2]);   /* K5 rank sums, K6 population groups */
int         bv_last_list_kernel_time(bv_ctx* ctx, float* ms);      /* K8 (bv_list_kernel, or bv_list_packed_kernel for compact
                                                                    * sparse lists) of the last lists tile */
int         bv_last_ranksum_kernel_time(bv_ctx* ctx, float* ms);   /* K9 bv_ranksum_test_kernel of the last bv_ranksum_test */

/* ---- tile pipeline (replaces: BatchInfo -> BaseType ctor -> lrt() -> strand_bias per site) ------ */
/* Asynchronous.  Host tiles are copied H2D on the slot's stream (pinned memory makes the copy truly
 * asynchronous), the kernels run, and the records are copied back to pinned staging.  A qual plane in
 * pinned memory (bv_host_alloc / cudaHostAlloc / cudaHostRegister) is not uploaded: the kernels read the
 * rows they need (those whose result depends on base qualities, ~10 % at 0.1x) in place over PCIe.
 * Host planes must stay valid and unchanged until bv_tile_wait() returns. */
int bv_tile_submit(bv_ctx* ctx, int slot, const bv_tile* tile);
/* Blocks until the slot is done and copies n_sites records to `out` (host memory). */
int bv_tile_wait(bv_ctx* ctx, int slot, bv_site_out* out);

/* For a tile submitted with out_mode == BV_OUT_COMPACT: blocks until the slot is done; *brief receives n_sites entries,
 * *full the *n_full full records they point into.  Both arrays are pinned staging of the slot (the records were written
 * there by the device): valid until the slot's next submit, no copy is made. */
int bv_tile_wait_compact(bv_ctx* ctx, int slot, const bv_site_brief** brief, const bv_site_out** full, uint32_t* n_full);
/* The record of a site whose brief has bit 31 of w0 clear (plain C, no CUDA).  ref_base: the site's REF character as
 * given in the tile; min_af: bv_params::min_af. */
void bv_site_expand(const bv_site_brief* brief, uint8_t ref_base, float min_af, bv_site_out* out);

/* Device-resident path: planes AND the output buffer are device pointers; nothing is copied.
 * `stream` is a cudaStream_t (NULL = the legacy default stream).  Stream ordered, returns at once. */
int bv_tile_run_device(bv_ctx* ctx, const bv_tile* tile, bv_site_out* d_out, void* stream);

/* ---- sparse host tiles: only the covered cells cross PCIe ------------------------------------------ */
/* At the depths this caller is built for (< 1x) nine cells in ten are the constant "uncovered" triple
 * (BV_BASE_N, phred 0, BV_STRAND_NONE) -- the `N ! 0 0 .` filler of the reference's batchfile rows
 * (src/basetype_caller.cpp:1063-1075).  A sparse tile carries the covered cells only, 4 bytes each, grouped by
 * site; the expand kernel (K0 bv_expand_kernel) writes the dense site-major planes in HBM and the same kernels
 * run on them, so the records are byte-identical with those of the dense tile.  Pileup assembly produces this
 * form naturally (one cell per aligned base of a read).
 *
 * cell = sample | base << 20 | strand << 23 | phred << 25   (sample < 2^20, base BV_BASE_*, strand BV_STRAND_*,
 * phred 0..127).  Within a site every sample index may appear at most once (first-read-wins has already been
 * applied by the packer); cells with sample >= n_samples, or offsets that are not ascending, make bv_tile_wait
 * fail with BV_ERR_ARG. */
#define BV_CELL_SAMPLE_BITS 20
#define BV_CELL_MAX_SAMPLES (1u << BV_CELL_SAMPLE_BITS)
#define BV_CELL_PACK(sample, base, strand, phred) \
    ((uint32_t)(sample) | ((uint32_t)(base) << 20) | ((uint32_t)(strand) << 23) | ((uint32_t)(phred) << 25))
/* aux word of a cell (called-site kernels): mapq | rpr << 8 */
#define BV_CELL_AUX_PACK(mapq, rpr) ((uint32_t)(mapq) | ((uint32_t)(rpr) << 8))

/* Compact form, 2 bytes per covered cell (BV_CELLS_U16): the words of a site in ASCENDING sample order,
 *   word = gap | base << 5 | strand << 8 | phred << 9      (gap 0..30, base BV_BASE_*, strand 0 '+' / 1 '-', phred 0..127)
 * where the cell's sample index = (index of the site's previous cell, or -1) + 1 + gap; a word with gap == 31 is no
 * cell but "skip 31 samples" (its other bits are 0).  At 0.1x the mean gap is 9 and one word in 25 is a skip.  A cell
 * whose strand is neither '+' nor '-' cannot be written this way (bv_sparse_encode16 says so; send the tile as
 * BV_CELLS_U32).  cells_aux, when used, is indexed like the words (the aux word of a skip is ignored). */
#define BV_CELLS_U32 0
#define BV_CELLS_U16 1
#define BV_CELL16_GAP_SKIP 31u
#define BV_CELL16_PACK(gap, base, strand, phred) \
    ((uint16_t)((uint32_t)(gap) | ((uint32_t)(base) << 5) | ((uint32_t)(strand) << 8) | ((uint32_t)(phred) << 9)))

typedef struct bv_sparse_tile {
    const void*     cells;      /* [site_start[n_sites]] words of `format`, the words of site 0 first: BV_CELL_PACK u32   */
                                /* (any order within a site) or BV_CELL16_PACK u16 (ascending samples)                     */
    const uint32_t* cells_aux;  /* same indexing, BV_CELL_AUX_PACK words; only read by bv_tile_submit_sparse_calls */
    const uint32_t* site_start; /* [n_sites + 1] ascending offsets into `cells`, in words; site_start[0] == 0     */
    const uint8_t*  ref_base;   /* [n_sites] as in bv_tile                                                        */
    bv_site_out*    out;        /* optional: PINNED host memory for the n_sites records; the D2H DMA then writes  */
                                /* them in place and bv_tile_wait's `out` may be NULL                             */
    uint32_t n_sites;
    uint32_t n_samples;
    uint32_t format;            /* BV_CELLS_U32 or BV_CELLS_U16                                                     */
    uint32_t out_mode;          /* BV_OUT_RECORDS, or BV_OUT_COMPACT (`out` must be NULL; collect with bv_tile_wait_compact) */
} bv_sparse_tile;

/* Asynchronous, like bv_tile_submit (host memory only; pinned memory makes the copies truly asynchronous). */
int bv_tile_submit_sparse(bv_ctx* ctx, int slot, const bv_sparse_tile* tile);
/* The same plus the called-site kernels; collect with bv_tile_wait_calls, or with bv_tile_wait_calls_compact when
 * out_mode is BV_OUT_COMPACT. */
int bv_tile_submit_sparse_calls(bv_ctx* ctx, int slot, const bv_sparse_tile* tile);
/* The same as bv_tile_submit_sparse plus lrt(list) per site (K8 on the planes K0 expanded, after the standard kernels); the
 * records are the bytes bv_tile_submit_sparse gives.  lists: n_sites x 4 bytes in host memory, read during the call, checked
 * as bv_tile_submit_lists checks them (BV_ERR_ARG, nothing submitted, the slot stays free).  Either cell format.
 *   out_mode BV_OUT_RECORDS: collect with bv_tile_wait_lists, one bv_lrt_out per site;
 *   out_mode BV_OUT_COMPACT: only the sites whose list is non-empty travel, 8 bytes up ({site, list}) and one bv_lrt_out
 *                            down each, packed in site order; collect with bv_tile_wait_lists_compact.
 * cells_aux is not read: lists and the called-site kernels do not run in one submit. */
int bv_tile_submit_sparse_lists(bv_ctx* ctx, int slot, const bv_sparse_tile* tile, const uint8_t (*lists)[4]);
/* For a lists tile with BV_OUT_COMPACT: blocks; brief / full / n_full as bv_tile_wait_compact gives them; lrt_out receives
 * *n_lrt entries, entry k belonging to the k-th site (in site order) whose list is non-empty.  BV_ERR_ARG (nothing copied to
 * lrt_out) when *n_lrt exceeds max_lrt. */
int bv_tile_wait_lists_compact(bv_ctx* ctx, int slot, const bv_site_brief** brief, const bv_site_out** full, uint32_t* n_full,
                               bv_lrt_out* lrt_out, uint32_t max_lrt, uint32_t* n_lrt);
/* BV_CELLS_U32 -> BV_CELLS_U16 on the host (plain C loop): the cells of every site must ascend by sample.  words16 has
 * room for max_words words (bv_sparse_encode16_bound() is always enough; pass words16 == NULL to count only);
 * start16[n_sites + 1] receives the word offsets, *n_words the word count.  BV_ERR_ARG: cells not ascending, a strand
 * that is neither '+' nor '-', or max_words too small.  aux16 (optional, with aux32) receives the aux words re-indexed. */
uint64_t bv_sparse_encode16_bound(uint64_t n_cells, uint32_t n_sites, uint32_t n_samples);
int bv_sparse_encode16(const uint32_t* cells, const uint32_t* aux32, const uint32_t* site_start, uint32_t n_sites,
                       uint16_t* words16, uint32_t* aux16, uint64_t max_words, uint32_t* start16, uint64_t* n_words);
/* Host twin of the synthetic generator in sparse form: fills cells / cells_aux (may be NULL) / site_start / ref_base
 * for sites [site0, site0 + n_sites); *n_cells receives the number of cells, BV_ERR_ARG if it exceeds max_cells
 * (call with cells == NULL to count only). */
int bv_synth_fill_sparse_host(const bv_synth_model* model, uint64_t site0, uint32_t n_sites, uint32_t n_samples,
                              uint32_t* cells, uint32_t* cells_aux, uint64_t max_cells, uint32_t* site_start,
                              uint8_t* ref_base, uint64_t* n_cells);

/* ---- called sites: rank-sum INFO fields and population-group allele frequencies ----------------- */
/* sample_group[i] = group index 0..n_groups-1 of sample i, or BV_GROUP_NONE.  The caller numbers the groups in the
 * order the reference iterates them (std::map<std::string,...>: ascending group name, basetype_caller.cpp:756).
 * n_groups == 0 turns the group kernel off.  Not allowed while a slot is busy. */
int bv_set_groups(bv_ctx* ctx, const uint8_t* sample_group, uint32_t n_samples, uint32_t n_groups);
/* bv_tile_submit + the kernels of the called sites.  `aux` planes live where the tile lives (host or device);
 * pageable host planes are uploaded whole, pinned ones are read in place for the called rows only.  Host tiles may ask for
 * BV_OUT_COMPACT (collect with bv_tile_wait_calls_compact); a device-resident tile that asks for it is refused (BV_ERR_ARG):
 * there is no device-resident compact form. */
int bv_tile_submit_calls(bv_ctx* ctx, int slot, const bv_tile* tile, const bv_tile_aux* aux);
/* Blocks; `out` receives n_sites records, `calls` up to max_calls entries, `groups` (may be NULL when no groups are
 * set) n_groups entries per call, groups[k * n_groups + g] belonging to calls[k].  *n_calls = number of called sites
 * of the tile; BV_ERR_ARG (nothing copied to calls/groups) when it exceeds max_calls. */
int bv_tile_wait_calls(bv_ctx* ctx, int slot, bv_site_out* out, bv_call_out* calls, uint32_t max_calls,
                       uint32_t* n_calls, bv_group_out* groups);
/* For a called-site tile with BV_OUT_COMPACT: blocks; brief / full / n_full as bv_tile_wait_compact gives them, calls / n_calls /
 * groups as bv_tile_wait_calls.  A called site is never all-REF, so its record is always among `full`; bv_call_out::site is the
 * site's row index, as in records mode. */
int bv_tile_wait_calls_compact(bv_ctx* ctx, int slot, const bv_site_brief** brief, const bv_site_out** full, uint32_t* n_full,
                               bv_call_out* calls, uint32_t max_calls, uint32_t* n_calls, bv_group_out* groups);
/* Device-resident variant (tile, aux planes, d_out, d_calls [n_sites], d_groups [n_sites * n_groups] and d_n_calls
 * are device pointers; d_groups may be NULL when no groups are set).  Stream ordered.  out_mode must be BV_OUT_RECORDS. */
int bv_tile_run_device_calls(bv_ctx* ctx, const bv_tile* tile, const bv_tile_aux* aux, bv_site_out* d_out,
                             bv_call_out* d_calls, bv_group_out* d_groups, uint32_t* d_n_calls, void* stream);

/* ---- lrt(specific_bases): per-site ordered candidate lists ----------------------------------------------- */
/* bv_tile_submit + the list kernel (K8 bv_list_kernel), which runs after the standard kernels and reads the depths and
 * strand counts of their records.  The records are the same bytes a plain bv_tile_submit gives.  lists: n_sites x 4
 * bytes in host memory, read during the call.  BV_ERR_ARG (nothing submitted, the slot stays free) for a repeated
 * base or a code that is neither BV_BASE_A..T nor BV_LIST_END.  Dense tiles with out_mode BV_OUT_RECORDS only (sparse tiles,
 * also with compact results: bv_tile_submit_sparse_lists).  Lists and the called-site kernels do not run in one submit:
 * bv_tile_wait_calls / bv_tile_wait_calls_compact on a lists slot return BV_ERR_STATE. */
int bv_tile_submit_lists(bv_ctx* ctx, int slot, const bv_tile* tile, const uint8_t (*lists)[4]);
/* Blocks; `out` receives n_sites records (may be NULL), `lrt_out` n_sites bv_lrt_out entries. */
int bv_tile_wait_lists(bv_ctx* ctx, int slot, bv_site_out* out, bv_lrt_out* lrt_out);
/* Device-resident variant: tile planes, d_lists [n_sites][4] (4-byte aligned), d_out and d_lrt_out are device pointers.
 * Stream ordered, so the lists are not seen before the kernel runs: a list the host entry points would refuse is treated
 * as an empty one here (all-zero entry).  out_mode must be BV_OUT_RECORDS (there is no device-resident compact form). */
int bv_tile_run_device_lists(bv_ctx* ctx, const bv_tile* tile, const uint8_t (*d_lists)[4], bv_site_out* d_out,
                             bv_lrt_out* d_lrt_out, void* stream);

/* ---- synthetic pileups --------------------------------------------------------------------------- */
int bv_synth_set_model(bv_ctx* ctx, const bv_synth_model* model);
/* Fill device planes for sites [site0, site0+n_sites) of the synthetic genome; mapq may be NULL. */
int bv_synth_fill_device(bv_ctx* ctx, uint64_t site0, uint32_t n_sites, uint32_t n_samples, uint64_t pitch,
                         uint8_t* d_base, uint8_t* d_qual, uint8_t* d_strand, uint8_t* d_mapq,
                         uint8_t* d_ref_base, void* stream);
/* Read-position-rank plane of the same synthetic genome (1 + draw % 35 for covered cells, 0 otherwise). */
int bv_synth_fill_rpr_device(bv_ctx* ctx, uint64_t site0, uint32_t n_sites, uint32_t n_samples, uint64_t rpr_pitch,
                             uint16_t* d_rpr, void* stream);
int bv_synth_fill_rpr_host(const bv_synth_model* model, uint64_t site0, uint32_t n_sites, uint32_t n_samples,
                           uint64_t rpr_pitch, uint16_t* rpr);
/* Host twin of the generator (plain C loop, no CUDA): same bytes as bv_synth_fill_device. */
int bv_synth_fill_host(const bv_synth_model* model, uint64_t site0, uint32_t n_sites, uint32_t n_samples,
                       uint64_t pitch, uint8_t* base, uint8_t* qual, uint8_t* strand, uint8_t* mapq,
                       uint8_t* ref_base);

/* ---- strand-bias statistic of arbitrary 2x2 tables ------------------------------------------------ */
/* strand_bias() (src/basetype.cpp:244-295) takes ANY set of ALT bases; the records carry FS for the two sets the caller
 * asks for (all non-REF bases: CVG row; the called ALT alleles: VCF row).  For any other set the 2x2 table follows from the
 * record's per-base strand counts and this call computes its FS on the device with the code of kernel KF, bv_fisher_kernel (two-sided Fisher
 * exact test restated from htslib/kfunc.c:245-313, FS rule src/basetype.cpp:277-283).  tables: n x {ref_fwd, ref_rev,
 * alt_fwd, alt_rev} in host memory, every table's total <= bv_params::max_samples + 1; fs_out: n doubles (host).
 * Blocking; a table with an empty row gives 0 (one possible outcome, p == 1). */
int bv_fisher_fs(bv_ctx* ctx, const int32_t* tables, uint32_t n, double* fs_out);

/* ---- rank-sum test of arbitrary REF / ALT classes ---------------------------------------------------------- */
/* ref_vs_alt_ranksumtest (src/basetype.h:168-176, src/basetype.cpp:201-242) for n free-standing problems, on the device.
 * Problem p: entries [start[p], start[p+1]) of bases (BV_BASE_* codes) and values; ref_base[p] raw ASCII (upper-cased as the
 * tile's REF is); alt_mask[p] bit b = base code b is an ALT.  phred_out[p]: the function's double, not truncated.
 * An entry whose base code is above BV_BASE_T is in neither class; one equal to the upper-cased REF is a REF read (whatever
 * the mask says); otherwise it is an ALT read when its bit is set.  The value is -10 log10 of the two-sided p of the Wilcoxon
 * rank-sum test (normal approximation, no tie correction, kf_erfc), 10000 when a class is empty or p == 0; a zero keeps the
 * sign the arithmetic gives (-0.0 when every value ties).  Exact for any int32 values.
 * Host memory, blocking.  BV_ERR_ARG (checked before anything is queued): null pointer (bases and values may be null when
 * start[n] == 0), start[0] != 0 or not ascending, a problem longer than max_samples, alt_mask > 15.  Nothing is launched for
 * n == 0. */
int bv_ranksum_test(bv_ctx* ctx, const uint8_t* bases, const int32_t* values, const uint64_t* start,
                    const uint8_t* ref_base, const uint8_t* alt_mask, uint32_t n, double* phred_out);

/* ---- tile sizing --------------------------------------------------------------------------------- */
/* The count kernel is persistent: num_SMs x W warps take one site row each (W = 32, or 16 for rows longer than 4,096
 * samples), so a tile whose site count is not a multiple of that leaves warps idle in the last round -- 16 % of the kernel
 * for 10,000 rows of 100,000 samples.  Returns the largest such multiple whose three planes (n_sites x round16(n_samples)
 * bytes each) fit max_bytes; when not even one multiple fits, the number of sites that do (at least 1). */
uint32_t bv_suggest_tile_sites(const bv_ctx* ctx, uint32_t n_samples, uint64_t max_bytes);

/* ---- pinned host memory helpers (for the packer / staging buffers of the caller) ---------------- */
int bv_host_alloc(void** out_ptr, size_t bytes);   /* cudaHostAlloc */
int bv_host_free(void* ptr);

#ifdef __cplusplus
}
#endif
#endif /* BASEVAR_B200_H */
