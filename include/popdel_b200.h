/* popdel_b200.h -- C ABI of the B200-native `popdel call` window scan.
 *
 * Drop-in boundary (SURVEY.md 8b, DESIGN.md "Boundary"): the reference has no FFI; its hot path is entered through
 *   (i)  ChromosomeProfile::add(rg, startPos, endPos, deviation)      popdel_call/profile_structure_popdel_call.h:1084-1113
 *        called from addRgRecordsToProfile                            popdel_call/load_profile_popdel_call.h:463-480
 *   (ii) processSegment(chromosomeProfile, calls, ...)                workflow_popdel.h:28-54, whose product is the
 *        String<Call> of window calls before unifyCalls               workflow_popdel.h:48
 * This library replaces both at contig granularity: pd_contig_begin = ChromosomeProfile::resetTo (window grid and
 * segment borders), pd_contig_push = the add() loop of one read group, pd_contig_scan = every processSegment() loop
 * of the contig (genotype_deletion_window for each 30-bp window). All functions return 0 on success or a negative
 * pd_status; no exception crosses the ABI; errors are sticky per context and described by pd_last_error().
 * Plain pointers and sizes only. One pd_ctx per GPU, driven by one host thread at a time -- with one exception:
 * pd_contig_push / pd_contig_push_pinned / _compact / _compact32 / _device may be called concurrently for DIFFERENT read groups of
 * one context (the host packer of a read group touches only that read group's staging; errors are recorded under a lock).
 */
#ifndef POPDEL_B200_H_
#define POPDEL_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pd_ctx pd_ctx;

enum pd_status {
    PD_OK = 0,
    PD_ERR_ARG = -1,          /* invalid argument / call order */
    PD_ERR_CUDA = -2,         /* CUDA runtime error or no usable device (no CPU fallback exists) */
    PD_ERR_RANGE = -3,        /* value not representable in the packed layout (deviation, position) */
    PD_ERR_CAPACITY = -4,     /* an internal device buffer was too small even after growing */
    PD_ERR_ORDER = -5         /* read pairs of a read group not sorted by position */
};

/* PopDelCallParameters subset that reaches the scan (popdel_call/parameter_parsing_popdel_call.h:141-210). */
typedef struct {
    uint32_t iterations;           /* -t, default 15 */
    uint32_t min_len;              /* params.minLen (95th percentile of min_init_del_len unless -m) */
    double   min_lr;               /* params.minimumLikelihoodRatio (parameter_calculation_popdel_call.h:16-23) */
    double   min_sample_fraction;  /* -s, default 0.1 */
    uint32_t window_size;          /* 30 (only 30 is supported, like the reference's profile conversion) */
    uint32_t window_buffer;        /* -b, default 200000: segment length in bp */
    int32_t  somatic;              /* -C */
    int32_t  window_wise;          /* -n: position = windowPosition, endPosition = 0 */
} pd_params;

/* One read group = one processed Histogram (insert_histogram_popdel.h:19-79) plus its per-RG parameters. */
typedef struct {
    uint32_t sample;               /* index of the owning sample; read groups of a sample are contiguous and ordered */
    uint32_t median;
    uint32_t read_length;
    double   stddev;
    int32_t  offset;               /* insert size of values[0] */
    uint32_t len;                  /* number of values */
    const double * values;         /* processed histogram (pd_process_histogram); copied by pd_create */
    double   min_prob;
    uint32_t lower_quantile_dist;
    uint32_t upper_quantile_dist;
    uint32_t max_load;             /* params.maxLoad[rg]; 0xFFFFFFFF disables the cap */
    uint32_t min_init_del_len;     /* params.minInitDelLengths[rg] */
} pd_rg;

/* One window call = reference struct Call (utils_popdel.h:57-124) without its per-sample strings. */
typedef struct {
    uint32_t initial_length, iterations, deletion_length;
    uint32_t filter;               /* bit 2 (value 4): sample-number filter (utils_popdel.h:158-170, 707-717) */
    double   lr, frequency;
    uint32_t window_position;      /* currentPos - 1 */
    uint32_t position, end_position;
    uint32_t segment;              /* index of the reference's processSegment() call (0-based per contig) */
} pd_call;

typedef struct {
    uint64_t n_calls;
    const pd_call * calls;         /* ordered by (window, initial_length), library-owned pinned memory */
    const uint32_t * per_sample;   /* n_calls x n_samples x 13: PL[3] LAD[3] DAD[5] FL[2] */
    uint64_t n_windows;            /* windows scanned (sample x window evaluations = n_windows * n_samples) */
    uint64_t n_flagged_windows;    /* windows that passed the exact screen and entered the genotyping stage */
    uint64_t n_candidates;         /* (window, initial length) pairs run through the EM */
    uint64_t n_reads;              /* read pairs resident on the device for this contig */
    uint64_t algorithmic_bytes;    /* bytes the screen kernel must move: 4 per resident read-pair word (DESIGN.md) */
    uint64_t h2d_bytes, d2h_bytes; /* bytes copied host->device for this contig / device->host for this scan */
    uint64_t n_kernel_launches;    /* kernels of this library launched by this scan */
    float    ms_h2d, ms_screen, ms_genotype, ms_d2h, ms_total;   /* CUDA-event times on the library's stream */
    float    ms_stream;            /* the HBM-bound streaming kernel of the screen alone (k_stream) */
    /* pd_set_unify only: calls / per_sample hold the MERGED variants of every segment (segment order, then
     * position / length order like unifyCalls' output) */
    const uint32_t * significant_windows;   /* n_calls x Call::significantWindows (SWIN); NULL without pd_set_unify */
    uint64_t n_window_calls;       /* window calls before the merge (they stayed on the device) */
    float    ms_unify;
    float    ms_em;                /* the FIRST EM chunk's kernels alone (k_em_one, or k_em + k_final); the whole EM when */
    uint32_t n_em_pairs_timed;     /* the scan has one chunk (<= 16384 (window, length) pairs) */
    uint64_t n_screened_windows;   /* windows left after the second screen stage (= n_flagged_windows when it is off) */
    uint64_t n_known_pairs;        /* second stage: (window, sample) pairs whose Q3 was computed before the stage decided */
} pd_result;

/* Host: processHistogram(hist, 256, smoothing, pseudoCountFraction), insert_histogram_popdel.h:974-986, in place.
 * Returns min_prob; writes the 1%/99% quantile distances. Needs no GPU. */
double pd_process_histogram(double * values, uint32_t len, int32_t offset, uint32_t median, uint32_t read_length,
                            int smoothing, uint32_t pseudo_count_fraction, uint32_t * lower_q, uint32_t * upper_q);

/* Creates a context on CUDA device `device` and copies parameters and histogram tables to it.
 * Returns NULL when no CUDA device is usable (pd_create_error() tells why). */
pd_ctx * pd_create(const pd_params * params, uint32_t n_samples, uint32_t n_rg, const pd_rg * rgs, int device);
const char * pd_create_error(void);
/* Initialises the CUDA context of `device` (no pd_ctx needed). Optional: a caller that has host work to do first
 * (decoding profiles) can run this on another thread so that pd_create does not pay the ~0.5 s context creation.
 * Returns 0 or PD_ERR_CUDA. Thread-safe. */
int pd_device_warmup(int device);
void pd_destroy(pd_ctx * ctx);
const char * pd_last_error(pd_ctx * ctx);

/* = ChromosomeProfile::resetTo(anchor) (profile_structure_popdel_call.h:1717-1748): starts a contig / region of
 * interest whose window grid is anchor + 30*i and whose segment borders are anchor + k*window_buffer. */
int pd_contig_begin(pd_ctx * ctx, uint32_t anchor);

/* = the ChromosomeProfile::add() calls for `n` read pairs of read group `rg`, in file order (sorted by position).
 * pos = reference end of the forward read, dev = insert size - median. Applies the active-coverage cap.
 * May be called several times per read group (positions must keep increasing). Host buffers are reusable on return. */
int pd_contig_push(pd_ctx * ctx, uint32_t rg, uint64_t n, const uint32_t * pos, const int32_t * dev);

/* Staging memory of pd_contig_push: page-locked (pinned != 0, the default: right for a context that uploads many
 * contigs, the buffers are reused) or pageable (pinned == 0: right for a one-shot caller such as the command-line shell,
 * for which page-locking a gigabyte once costs more than the slower pageable copy). Applies to buffers allocated
 * afterwards. */
int pd_set_staging(pd_ctx * ctx, int pinned);
/* Fast path of pd_contig_push for PAGE-LOCKED host arrays (cudaHostAlloc / cudaHostRegister / torch pin_memory):
 * the library only records the pointers; pd_contig_upload copies the raw arrays to the device and packs them THERE
 * (tile search, scan, words, wide list). The arrays must stay valid and unchanged until pd_contig_upload (or the
 * first pd_contig_scan) returns. One call per read group and contig; cannot be mixed with pd_contig_push. Same
 * results as pd_contig_push: the active-coverage cap is checked exactly on the device and, if it would drop a read
 * pair, the contig is transparently re-packed by the sequential host path. */
int pd_contig_push_pinned(pd_ctx * ctx, uint32_t rg, uint64_t n, const uint32_t * pos, const int32_t * dev);

/* pd_contig_push_pinned with 5 instead of 8 bytes per read pair over PCIe (the profile file stores 5: a u8 offset inside
 * its 256-bp window and an i32 deviation, window_podel.h:161-197): positions are split into 65 536-bp blocks,
 *   blk_first[b]  index of the first read pair with pos >> 16 == b, b = 0 .. n_blocks (blk_first[n_blocks] = n),
 *   pos_lo[i]     pos & 0xFFFF,
 *   dev24[3 * i]  the deviation as a little-endian two's-complement 24-bit integer (|dev| < 2^20 in the packed layout).
 * The arrays are expanded on the device. Same rules as pd_contig_push_pinned (page-locked, valid until the upload
 * returns, one call per read group and contig, identical results). */
int pd_contig_push_compact(pd_ctx * ctx, uint32_t rg, uint64_t n, const uint16_t * pos_lo, const uint8_t * dev24,
                           uint32_t n_blocks, const uint32_t * blk_first);

/* The densest input form, 4 bytes per read pair (+ 4 bytes per 256-bp block): word[i] = deviation << 8 | (pos & 0xFF) with
 * the deviation as a 24-bit two's-complement integer, and blk_first[b] = index of the first read pair with pos >> 8 == b,
 * b = 0 .. n_blocks (blk_first[n_blocks] = n) -- the layout of the profile file itself (a u8 offset inside its 256-bp window,
 * window_podel.h:161-197). Same rules and results as pd_contig_push_compact. */
int pd_contig_push_compact32(pd_ctx * ctx, uint32_t rg, uint64_t n, const uint32_t * words, uint32_t n_blocks, const uint32_t * blk_first);

/* pd_contig_push_pinned for arrays that are ALREADY in the memory of the context's GPU (written there by a device-side
 * profile decoder or generator): pos / dev are device pointers; nothing crosses PCIe, the arrays are packed where they
 * are. Same rules (valid until the upload returns, one call per read group and contig, may be mixed with
 * pd_contig_push_pinned / _compact for other read groups, identical results; if the active-coverage cap would drop a read
 * pair the arrays are copied to the host once and re-packed by the sequential host path). */
int pd_contig_push_device(pd_ctx * ctx, uint32_t rg, uint64_t n, const uint32_t * d_pos, const int32_t * d_dev);

/* Packs what was pushed and copies it to the device (pinned staging, async on the context's stream). */
int pd_contig_upload(pd_ctx * ctx);

/* = all processSegment() window loops of the contig: scans windows [first_window, first_window + n_windows)
 * (n_windows = 0: up to the reference's last scanned window) over the device-resident read pairs and returns the
 * window calls. Uploads first if needed. `out` stays valid until the next call on this context. */
int pd_contig_scan(pd_ctx * ctx, uint64_t first_window, uint64_t n_windows, pd_result * out);

/* = unifyCalls(calls, meanStddev, minRelWinCover, outputFailed) per processSegment() call (utils_popdel.h:567-654,
 * workflow_popdel.h:48) ON THE DEVICE: after pd_set_unify(ctx, &p) every pd_contig_scan keeps its window calls and
 * their per-sample rows in device memory, merges the windows of every segment into variants there (sort by position /
 * length / LR, chain of similar calls, median start and length, PLs summed over the variant's windows and
 * re-normalised, median LAD / DAD, allele frequency from the genotypes, CSWin filter bit 16) and returns only the
 * merged variants. Segments with a single window call, or without a passing one (unless output_failed), return
 * nothing, like the reference. pd_set_unify(ctx, NULL) switches back to window calls. May be called before or after
 * attaching a context to a sample-sharded cohort; every rank must then use the same settings (a collective scan whose ranks
 * differ fails with PD_ERR_ARG on every rank before any kernel runs). Each rank returns the same merged variants, with
 * the allele frequency over all n_samples_global samples, and per_sample holds the merged rows of its own samples. */
typedef struct {
    double  mean_stddev;                   /* mean insert-size standard deviation over all read groups */
    double  min_relative_window_cover;     /* -c, default 0.5 */
    int32_t output_failed;                 /* -F */
    int32_t reserved;
} pd_unify_params;
int pd_set_unify(pd_ctx * ctx, const pd_unify_params * p);
/* Sizes the tile tables of the open contig for at least `n_windows` windows (call between pd_contig_begin and the
 * upload). Needed by sample-sharded cohorts, whose ranks must cover the COHORT's window range (normally contig length
 * / 30 + 2) although their own samples' read pairs may end earlier. */
int pd_contig_reserve_windows(pd_ctx * ctx, uint64_t n_windows);

/* ---- Sample sharding (SURVEY.md 8e; BASELINE.json: "only the largest-cohort config additionally shards by sample") ----
 * Every rank creates its context with ITS samples / read groups only (pd_create) and attaches it to the cohort:
 * the screen threshold, the rank-indexed initial-length thresholds (initialize_deletion_lengths,
 * genotype_deletion_popdel_call.h:58-86), the sample count of update_allele_frequency (:467-485) and of the
 * sample-fraction filter become the cohort's; read group 0 of the COHORT drives every reference shift (:401,424-431).
 * pd_contig_scan is then a COLLECTIVE: all ranks call it with the same window range after pushing their read pairs
 * (and pd_contig_reserve_windows). It all-gathers the screen's tile flags, the per-window Q3 values and the contig
 * tail, and exchanges the EM's per-iteration sufficient statistics inside the EM kernels through peer memory
 * (NVLink). Every rank returns the same calls; per_sample holds the rows of the rank's own samples. With pd_set_unify
 * on every rank the window calls stay on the devices: each rank merges them over its own samples and the ranks
 * all-gather one allele count per merged variant for the frequency. */
typedef struct {
    uint32_t rank, world;                  /* world = 2..8 */
    uint32_t n_samples_global;
    uint32_t n_rg_global;
    const uint32_t * min_init_global;      /* [n_rg_global] minInitDelLengths of all read groups, cohort order */
    const uint32_t * samples_per_rank;     /* [world]; rank r holds the samples after those of ranks < r */
} pd_shard_info;

/* One process per GPU: NCCL (all-gathers) + CUDA IPC (exchange slots). Rank 0 makes the 128-byte id, the launcher
 * distributes it (e.g. torch.distributed.broadcast), every rank attaches (collective). libnccl.so.2 is dlopen'ed. */
int pd_shard_unique_id(uint8_t * out128);
int pd_shard_attach_nccl(pd_ctx * ctx, const pd_shard_info * info, const uint8_t * id128);

/* Several contexts of ONE process (on one GPU or on peer-accessible GPUs): infos[r] describes rank r.
 * pd_shard_group_scan runs the collective scan with one host thread per context. */
int pd_shard_attach_group(pd_ctx ** ctxs, uint32_t n, const pd_shard_info * infos);
int pd_shard_group_scan(pd_ctx ** ctxs, uint32_t n, uint64_t first_window, uint64_t n_windows, pd_result * outs);

/* Number of grid windows the reference would scan for the pushed contig (last scanned window index + 1). */
int pd_contig_window_count(pd_ctx * ctx, uint64_t * n_windows);

/* Host-side validation hook for the packed layout (NOT used by the scan): per-window active read-pair count,
 * sum of deviations and sum of positions of read group `rg`, computed from the packed words with the same
 * closed-form activity rule the kernels use. out = n_windows x 3 int64. Needs no GPU. */
int pd_debug_host_window_sums(pd_ctx * ctx, uint32_t rg, uint64_t first_window, uint64_t n_windows, int64_t * out);

/* Host-side validation hook for the active-coverage cap of pd_contig_push (ChromosomeProfile::add,
 * profile_structure_popdel_call.h:1084-1113): stored[i] = 1 when read pair i (anchor-relative start position and
 * end = start + max(0, inner distance), sorted by start) of a read group with cap max_load is kept. Needs no GPU. */
int pd_debug_cap_replay(uint32_t window_buffer, uint32_t max_load, uint64_t n, const uint32_t * start, const uint32_t * end,
                        uint8_t * stored);

#ifdef __cplusplus
}
#endif
#endif /* POPDEL_B200_H_ */
