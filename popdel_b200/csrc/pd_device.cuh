// pd_device.cuh -- device-side helpers and the kernel-launch interface shared by the scan's translation units
// (pd_screen.cu, pd_gather.cu, pd_em.cu, pd_scan.cu). Internal.
#ifndef PD_DEVICE_CUH_
#define PD_DEVICE_CUH_

#include <climits>
#include <string>

#include "pd_context.h"

#define PD_CUDA(c, call)                                                                          \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess)                                                                    \
            return pd_fail((c), PD_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

#define PD_MAX_WORLD 8                              /* ranks of a sample-sharded cohort */
constexpr uint32_t PD_FULL = 0xFFFFFFFFu;
constexpr uint32_t PD_GRAN = 1024;                  // words per warp in k_stream; granule of the word -> tile index
constexpr int PD_CAND_INLINE = 6;                   // candidate lengths kept inline per window job
constexpr uint32_t PD_GRID_Y_MAX = 65535;           // CUDA's limit on gridDim.y and gridDim.z
constexpr uint32_t PD_CAND_SMEM = 202 * 1024;       // bytes of Q3s k_candidates keeps in shared memory (one int per sample)

// Launches over `rows` samples or read groups: gridDim.y is capped, gridDim.z takes the rest; the block's row is
// pd_grid_row() (rows up to 65 535^2; blocks past the last row exit)
inline dim3 pd_rows_grid(uint32_t x, uint32_t rows)
{
    const uint32_t y = rows < PD_GRID_Y_MAX ? (rows ? rows : 1u) : PD_GRID_Y_MAX;
    return dim3(x, y, (rows + y - 1) / y);
}

// device counters of one scan (uint32 each)
enum { CNT_TJOBS = 0, CNT_JOBS = 1, CNT_PAIRS = 2, CNT_POOL = 3, CNT_CALLS = 4, CNT_CJOBS = 5, CNT_ERR = 6, CNT_ALIVE = 7, CNT_KNOWN = 8, CNT_KJOBS = 9, CNT_N = 16 };

struct PdPair { uint32_t job; int32_t L0; };                         // (window job, initial deletion length)
struct EmState { uint32_t len, it, alive, pad; double freq; double gt[3]; };   // handed from k_em to k_final

// ---- screen (pd_screen.cu) ------------------------------------------------------------------------------------
struct ScreenArgs {
    uint32_t tile_begin, tile_end;      // tiles intersecting the window range
    uint32_t tb_al;                     // tile_begin rounded down to a multiple of 32
    uint32_t need_stride;               // words of the need bitmap per sample
    uint32_t * need;                    // [N][need_stride] bit = (sample, tile) can see a read pair above the threshold
    uint32_t * tile_flags;              // [tile_end - tile_begin] bit = window of the tile passed the exact screen
    const uint32_t * gran_off;          // [R+1] first entry of read group g in gran_tile
    const uint32_t * gran_tile;         // tile that contains word (first word of g) + j * PD_GRAN
    const uint32_t * long_off;          // [R+1] wide-list ranges per read group
    uint32_t total_longs;
    uint32_t * known;                   // second stage: [N][need_stride * 32] window bits per (sample, tile): Q3 can exceed t_known
    uint2 * kjobs; uint32_t kjobs_cap;  // second stage: the (sample, tile) pairs that have such windows (counters[CNT_KJOBS] of them, any order)
    uint32_t * counters;
};
struct JobArgs {
    const uint32_t * tile_flags; uint32_t n_tiles, tile_begin;
    uint32_t * tj_tile, * tj_mask, * tj_wbase;      // flagged tiles in ascending order, window mask, first window job
    uint32_t * job_window;                           // window of every window job (ascending)
    uint32_t * tj_of_tile;                           // [n_tiles] tile job of a flagged tile (0xFFFFFFFF: none); may be null
    uint32_t * counters;
    unsigned long long * block_sums;                // scratch of the two-level scan
};
void pd_launch_gran_index(const PdDev & a, uint32_t * gran_tile, const uint32_t * gran_off, cudaStream_t st);
void pd_launch_tile_segs(uint4 * out, uint32_t n, uint32_t window_buffer, cudaStream_t st);
void pd_launch_screen(const PdDev & a, const ScreenArgs & s, uint32_t max_rg_words, cudaStream_t st, cudaEvent_t after_stream, uint64_t * launches);
void pd_launch_tile_jobs(const JobArgs & j, cudaStream_t st, uint64_t * launches);
// pd_debug_device_window_sums: per-window count / sum of deviations / sum of positions of read group g, windows [w_first, w_end)
// of tiles [tile_begin, tile_end), as for_tile_batches walks them; out[3 * (w - w_first) + k]
void pd_launch_window_sums(const PdDev & a, uint32_t g, uint32_t anchor, uint32_t tile_begin, uint32_t tile_end, uint64_t w_first,
                           uint64_t w_end, unsigned long long * out, cudaStream_t st);

// ---- gather + candidates (pd_gather.cu) -----------------------------------------------------------------------
struct GatherArgs {
    const uint32_t * tj_tile, * tj_mask, * tj_wbase; uint32_t tj0, ntj;      // tile jobs [tj0, tj0 + ntj)
    uint32_t job_base;                  // first window job of this batch (scratch rows are relative to it)
    // Q3 pass (k_tile_q3): every flagged window
    int32_t * q3; uint8_t * sstat;      // [jobs][N]   sstat: 0 = low coverage, 1 = no usable values, 2 = Q3 valid
    int32_t * dmax;                     // [jobs][N]   largest deviation among the sample's usable active read pairs (INT_MIN: none)
    // pool pass (k_tile_gather): windows with candidate lengths ("candidate jobs", numbered in window order per batch)
    const uint32_t * tj_cmask, * tj_cfirst;      // [ntj] candidate windows of the tile / candidate job of the first of them
    uint32_t cj_base, cj_end;           // this launch handles the tiles whose first candidate job lies in [cj_base, cj_end)
    uint32_t * pool_pos; int32_t * pool_dev; uint32_t pool_cap;              // active read pairs, SoA
    uint32_t * counters;
    uint32_t * act_off, * act_cnt;      // [candidate jobs - cj_base][R]
    uint32_t debug_flags;               // tests: bit 0 = generic path in k_tile_q3, bit 1 = generic path in k_tile_gather
    // second screen stage (pd_launch_q3 phases): 0 = every (flagged window, sample); 1 = only the pairs whose Q3 can exceed
    // t_known; 2 = the rest, for the windows the stage could not reject
    int phase;
    const uint32_t * known; uint32_t known_stride, tb_al;
    const uint2 * kjobs; uint32_t n_kjobs;          // phase 1 walks this list of (sample, tile) instead of every (tile job, sample)
    const uint32_t * tj_of_tile; uint32_t tile_begin;
    uint32_t * tj_alive;                // [ntj] windows of the tile job that survive the second stage
    uint8_t * job_dead;                 // [jobs] 1 = rejected by the second stage (no candidates possible)
};
struct CandArgs {
    // Q3 / state of every (window job, sample): nparts blocks [njobs][part_n[p]] (one per rank when sharded by sample)
    uint32_t nparts; const int32_t * q3[PD_MAX_WORLD]; const uint8_t * sstat[PD_MAX_WORLD]; uint32_t part_n[PD_MAX_WORLD];
    const uint32_t * min_init;          // [read groups of the whole cohort] minInitDelLengths, indexed by RANK (quirk)
    uint32_t njobs, job_base;
    uint32_t * cand_cnt;                // [njobs]
    int32_t * cand_inline;              // [njobs][PD_CAND_INLINE]
    uint32_t * cand_off;                // [njobs] exclusive scan of cand_cnt
    uint32_t * cjob_of;                 // [njobs] number of earlier windows of the batch with candidates (= candidate job)
    PdPair * pairs; uint32_t pair_cap;
    uint32_t * counters; unsigned long long * block_sums;
    uint32_t npad;                      // samples of the cohort, rounded up to a multiple of 32
    uint32_t force_sort;                // tests: always take the sorting path of k_candidates
    const uint8_t * job_dead;           // second screen stage: windows without any possible candidate (nullptr: stage off)
    int32_t * sort_buf;                 // nullptr: k_candidates keeps the Q3s in shared memory; else [njobs][npad] for the
                                        // sorting fallback of the instance that reads them from global memory
};
void pd_launch_q3(const PdDev & a, const GatherArgs & g, cudaStream_t st, uint64_t * launches);
void pd_launch_screen2(const PdDev & a, const GatherArgs & g, cudaStream_t st, uint64_t * launches);
void pd_launch_cmask(const GatherArgs & g, const CandArgs & ca, uint32_t * tj_cmask, uint32_t * tj_cfirst, cudaStream_t st, uint64_t * launches);
void pd_launch_gather(const PdDev & a, const GatherArgs & g, cudaStream_t st, uint64_t * launches);
int  pd_launch_candidates(pd_ctx * c, const PdDev & a, const CandArgs & ca, cudaStream_t st, uint64_t * launches);

// ---- sample sharding (pd_shard.cu): cross-rank exchange inside the EM kernels --------------------------------------
// One slot = the four 64-bit values one rank contributes to one reduction of one (window, length) pair. Every rank
// owns an array [2 launches][pairs][2 reductions][world ranks]; rank r WRITES slot [..][r] of every rank's array
// (peer memory over NVLink, or plain device memory for in-process groups) and POLLS its own array.
struct XrSlot { unsigned long long v[4]; unsigned long long seq; unsigned long long pad[3]; };
struct XrArgs {
    uint32_t world, rank;               // world <= 1: not sharded
    XrSlot * peer[PD_MAX_WORLD];        // rank r's slot array
    uint32_t pairs_cap;                 // pairs per launch the arrays hold
    unsigned long long epoch;           // launch number, identical on every rank (sequence numbers = epoch << 16 | k)
    uint32_t * ticket;                  // pair numbering of the persistent launch
    uint32_t * err;                     // set when a peer did not answer in time (the scan then fails)
    uint32_t n_global;                  // samples of the whole cohort
    uint32_t owns_rg0;                  // this rank holds read group 0 of the cohort (its posterior drives every reference shift)
    uint32_t grid_cap;                  // blocks of the persistent launch
};

// ---- EM + final pass (pd_em.cu) -------------------------------------------------------------------------------
struct EmArgs {
    const uint32_t * job_window; const PdPair * pairs; uint32_t pair0, npairs, job_base;   // pairs[].job is absolute
    const uint32_t * pool_pos; const int32_t * pool_dev; const uint32_t * act_off, * act_cnt; const uint8_t * sstat;
    const int32_t * dmax;    // [job][N]
    const uint32_t * cjob_of; uint32_t cj_base;      // act_off / act_cnt rows: cjob_of[job] - cj_base
    double * dlx;            // [pair][N][3]   data likelihoods, log domain, max = 0
    double * dle;            // [pair][N][3]   exp(dlx)
    int32_t * shifts;        // [pair][R]
    uint32_t * ps;           // [pair][N][13]  per-sample output rows
    pd_call * calls;         // [pair]
    uint8_t * valid;         // [pair]
    uint32_t * done;         // [pair] set (release) when valid / calls / ps of the pair are final
    EmState * states;        // [pair]
    uint32_t iterations, min_len; double min_lr, min_sample_fraction; int somatic, window_wise; uint32_t anchor;
    uint32_t * dbg;          // optional [npairs][4]: reason, len, iterations, supp (PD_DEBUG)
    int dbg_window;          // device printf of the EM trajectory of this window (PD_DEBUG_WINDOW), -1 = off
    int sort_samples;        // fused kernel: order the samples by largest deviation and skip unchanged likelihood passes
    XrArgs xr;               // sample sharding: cross-rank reductions (world <= 1: none)
};
struct EmitArgs {
    const uint8_t * valid; const pd_call * calls; const uint32_t * ps; uint32_t npairs, row_words;
    const uint32_t * done;              // [pair] published by the EM kernels
    uint32_t * counters;                // CNT_CALLS = calls emitted so far, CNT_ERR = the emitter gave up waiting
    uint32_t * emit_blocks_done;        // device scalar (0 between launches)
    pd_call * out_calls; uint32_t * out_ps; uint32_t * out_count;   // mapped page-locked host memory
};
int  pd_launch_em(pd_ctx * c, const PdDev & a, const EmArgs & e, cudaStream_t st, uint64_t * launches);
// second-generation genotyping pipeline (pd_em2.cu): sample-major, likelihood tables in shared memory
enum { PD_S_E2_ITEM = 40, PD_S_E2_CTL, PD_S_E2_CUR, PD_S_E2_REC, PD_S_E2_RECA, PD_S_E2_STAT, PD_S_E2_INV, PD_S_E2_FIN, PD_S_E2_PST,
       PD_S_E2_BOFF, PD_S_E2_BNMAX, PD_S_E2_SUPPN, PD_S_E2_SUPPF, PD_S_E2_SUPPL, PD_S_E2_DEVT, PD_S_E2_POST, PD_S_E2_CNT, PD_S_E2_FLAGS, PD_S_E2_ACT, PD_S_END };
int  pd_grow_scratch(pd_ctx * c, int slot, size_t bytes, void ** p);      // pd_scan.cu
bool pd_em2_usable(const pd_ctx * c);
size_t pd_em2_pair_bytes(uint32_t R, double reads_per_pair);
int  pd_launch_em2(pd_ctx * c, const PdDev & a, const EmArgs & e, double reads_per_pair, cudaStream_t st, uint64_t * launches);
int  pd_em2_overflow(pd_ctx * c, bool * ovf, size_t * need_words);
int  pd_em_preload_xr(pd_ctx * c);
void pd_launch_emit(const EmitArgs & m, cudaStream_t st, uint64_t * launches);

#if defined(__CUDACC__)
// ---------------------------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pd_grid_row() { return blockIdx.z * gridDim.y + blockIdx.y; }      // see pd_rows_grid

__device__ __forceinline__ PdTile load_tile(const PdTile * p)
{
    const uint4 q = __ldg(reinterpret_cast<const uint4 *>(p));
    return PdTile{q.x, q.y, q.z, q.w};
}

// block-wide exclusive scan of one 64-bit value per thread (blockDim.x multiple of 32, <= 1024); returns the
// exclusive prefix, `total` = sum over the block. `ws` = 33 values of shared memory.
__device__ __forceinline__ unsigned long long block_excl_scan(unsigned long long v, unsigned long long * ws, unsigned long long & total)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    unsigned long long inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned long long n = __shfl_up_sync(PD_FULL, inc, o); if (lane >= o) inc += n; }
    __syncthreads();                                    // ws may still be read from a previous call
    if (lane == 31) ws[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        unsigned long long s = lane < nw ? ws[lane] : 0ull, si = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned long long n = __shfl_up_sync(PD_FULL, si, o); if (lane >= o) si += n; }
        if (lane < nw) ws[lane] = si - s;
        if (lane == 31) ws[32] = si;
    }
    __syncthreads();
    total = ws[32];
    return ws[wid] + inc - v;
}

// calls f(valid, s, e, pos_rel, dev) for every 32-wide batch of read pairs of read group g whose active interval can
// intersect the windows of `tile` (stream words of the look-back tiles in stream order, then the wide list).
// `valid` marks lanes holding a real, ever-active read pair; the caller tests the interval. Must be called by all 32
// lanes. The look-back tiles are contiguous in the stream: lane j holds the table entry and segment constants of tile
// t_lo + j (ONE load phase instead of one per tile), the words are walked as one flat range with the next batch
// already in flight, and every lane finds the tile of its word among the <= 9 tile borders by shuffles.
template <typename F>
__device__ __forceinline__ void for_tile_batches(const PdDev & a, uint32_t g, const PdRgConst & k, uint32_t tile, int lane, F f)
{
    const PdTile * tl = a.tiles + (size_t)g * (a.NT + 1);
    const uint32_t t_lo = tile > k.lookback_tiles ? tile - k.lookback_tiles : 0;
    const uint32_t nt = tile - t_lo + 1;                              // <= PD_MAX_LOOKBACK_TILES + 1
    PdTile mine = PdTile{0xFFFFFFFFu, 0, 0, 0};
    if ((uint32_t)lane <= nt) mine = load_tile(&tl[t_lo + lane]);
    // Only the tail of the look-back matters: tile t_lo + j is needed iff one of its read pairs reaches nt-1-j tiles ahead
    // (PdTile::reach, written by the packers); of the tile right before `tile` only the words from the first one that reaches over.
    const uint32_t ahead = nt - 1u - (uint32_t)lane;
    const uint32_t needed = __ballot_sync(PD_FULL, (uint32_t)lane + 1u < nt && (mine.reach >> 24) >= ahead);
    const int j_first = needed ? __ffs(needed) - 1 : (int)nt - 1;
    uint32_t r_lo = __shfl_sync(PD_FULL, mine.off + (((uint32_t)lane + 2u == nt) ? (mine.reach & 0xFFFFFFu) : 0u), j_first);
    const uint32_t r_hi = __shfl_sync(PD_FULL, mine.off, (int)nt);
    r_lo &= ~3u;                                                      // keep the 128-bit alignment of the tile starts
    const uint32_t l_lo = __shfl_sync(PD_FULL, mine.long_lo, (int)nt - 1), l_hi = __shfl_sync(PD_FULL, mine.long_hi, (int)nt - 1);
    // borders 1..3 in registers (warp-uniform); 0xFFFFFFFF beyond the look-back
    const uint32_t b1 = nt > 1 ? __shfl_sync(PD_FULL, mine.off, 1) : 0xFFFFFFFFu;
    const uint32_t b2 = nt > 2 ? __shfl_sync(PD_FULL, mine.off, 2) : 0xFFFFFFFFu;
    const uint32_t b3 = nt > 3 ? __shfl_sync(PD_FULL, mine.off, 3) : 0xFFFFFFFFu;
    // the segment constants of the look-back tiles differ only in base_bp unless a segment border lies between them
    // (tile_seg costs ~100 instructions: one 32-bit and three 64-bit divisions; the per-tile table is one 16-byte load)
    auto seg_of = [&](uint32_t t) {
        const uint4 q = __ldg(a.tseg + t);
        TileSeg s; s.base_bp = t * PD_TILE_BP; s.nb = q.x; s.wlA = (int32_t)q.y; s.wlB = (int32_t)q.z; s.wlC = (int32_t)q.w;
        return s;
    };
    const TileSeg ts_hi = seg_of(tile);
    const bool one_seg = nt == 1 || __ldg(&a.tseg[t_lo].x) == ts_hi.nb;
    uint32_t next = (r_lo + lane) < r_hi ? __ldg(a.words + r_lo + lane) : PD_PAD_WORD;
    for (uint32_t base = r_lo; base < r_hi; base += 32) {
        const uint32_t i = base + lane, word = next;
        if (base + 32 < r_hi) next = (i + 32) < r_hi ? __ldg(a.words + i + 32) : PD_PAD_WORD;
        uint32_t kk = (uint32_t)(i >= b1) + (uint32_t)(i >= b2) + (uint32_t)(i >= b3);      // tile of word i = t_lo + borders <= i
        for (uint32_t j = 4; j < nt; ++j) kk += __shfl_sync(PD_FULL, mine.off, (int)j) <= i;
        TileSeg ts = ts_hi;
        if (one_seg) ts.base_bp = (t_lo + kk) * PD_TILE_BP;
        else ts = seg_of(t_lo + kk);
        int32_t s = 0, e = 0, dev = 0; uint32_t pr = 0;
        const bool valid = word_interval(word, ts, k.inner_off, s, e, dev, pr);
        f(valid, s, e, pr, dev);
    }
    for (uint32_t base = l_lo; base < l_hi; base += 32) {
        const uint32_t i = base + lane;
        PdLong L = PdLong{0xFFFFFFFFu, 0, 0, 0};
        if (i < l_hi) L = a.longs[i];
        f(i < l_hi, (int32_t)L.s, (int32_t)L.e, L.pos_rel, L.dev);
    }
}
#endif  // __CUDACC__

#endif
