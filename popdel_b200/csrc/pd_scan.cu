// pd_scan.cu -- orchestration of one window-range scan (pd_contig_scan): screen -> tile jobs -> gather ->
// candidates -> EM / final pass in chunks -> ordered emission into mapped host memory.
//
// Host synchronisations per scan: one after the screen (number of flagged tiles / windows, to size the scratch), one
// per job batch after the candidates (number of (window, length) pairs), one at the end. Everything else is
// stream-ordered: the EM chunks run on `stream`, the emission of chunk k (k_emit_*, writing call headers and per-sample
// rows over PCIe) runs on `stream2` and overlaps the EM of chunk k+1.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "pd_device.cuh"
#include "pd_shard.h"

namespace {

enum Slot {                                     // d_scratch slots
    S_NEED = 0, S_TFLAGS, S_COUNTERS, S_TJ_TILE, S_TJ_MASK, S_TJ_WBASE, S_JOBWIN, S_BSUMS,
    S_ACT_OFF, S_ACT_CNT, S_Q3, S_SSTAT, S_CAND_CNT, S_CAND_INL, S_CAND_OFF, S_CJOB_OF, S_TJ_CMASK, S_TJ_CFIRST, S_PAIRS, S_POOL_POS, S_POOL_DEV,
    S_DLX, S_DLE, S_SHIFTS, S_STATES, S_PS0, S_PS1, S_CALLS0, S_CALLS1, S_VALID0, S_VALID1, S_DONE0, S_DONE1, S_CHUNK_BASE, S_DBG, S_DMAX, S_ALL_Q3, S_ALL_SS, S_CAND_SORT,
    S_KNOWN = 64, S_TJ_ALIVE, S_JOB_DEAD, S_KJOBS, S_TJ_OF_TILE
};

template <typename T>
int grow_scratch(pd_ctx * c, int slot, T *& p, size_t need)
{
    const size_t bytes = std::max<size_t>(need, 1) * sizeof(T);
    if (bytes > c->cap_scratch[slot] || !c->d_scratch[slot]) {
        if (c->d_scratch[slot]) cudaFree(c->d_scratch[slot]);
        c->d_scratch[slot] = nullptr; c->cap_scratch[slot] = 0;
        const size_t want = std::max<size_t>(bytes + bytes / 4, 4096);
        PD_CUDA(c, cudaMalloc(&c->d_scratch[slot], want));
        c->cap_scratch[slot] = want;
    }
    p = reinterpret_cast<T *>(c->d_scratch[slot]);
    return 0;
}

}  // namespace

int pd_grow_scratch(pd_ctx * c, int slot, size_t bytes, void ** p)
{
    uint8_t * q = nullptr;
    if (grow_scratch(c, slot, q, bytes)) return c->status;
    *p = q;
    return 0;
}

namespace {

// word -> tile index and wide-list ranges of the current upload (built once per upload)
int build_index(pd_ctx * c, PdDev & a)
{
    const uint32_t R = c->R;
    if ((size_t)c->NT + 1 > c->cap_tseg || !c->d_tseg) {
        cudaFree(c->d_tseg); c->d_tseg = nullptr; c->cap_tseg = 0;
        const size_t want = (size_t)c->NT + 1 + c->NT / 8;
        PD_CUDA(c, cudaMalloc(&c->d_tseg, want * sizeof(uint4)));
        c->cap_tseg = want;
    }
    pd_launch_tile_segs(c->d_tseg, c->NT + 1, a.window_buffer, c->stream);
    a.tseg = c->d_tseg;
    std::vector<uint32_t> goff(R + 1, 0);
    uint32_t max_words = 0;
    for (uint32_t g = 0; g < R; ++g) {
        const uint64_t nw = c->h_word_base[g + 1] - c->h_word_base[g];
        goff[g + 1] = goff[g] + (uint32_t)((nw + PD_GRAN - 1) / PD_GRAN) + 1;
        max_words = (uint32_t)std::max<uint64_t>(max_words, nw);
    }
    c->max_rg_words = max_words;
    const size_t need = (size_t)goff[R] + 1;
    if (need > c->cap_gran || !c->d_gran_tile) {
        cudaFree(c->d_gran_tile); cudaFree(c->d_gran_off); cudaFree(c->d_long_off);
        c->d_gran_tile = c->d_gran_off = c->d_long_off = nullptr; c->cap_gran = 0;
        PD_CUDA(c, cudaMalloc(&c->d_gran_tile, (need + need / 8) * 4));
        PD_CUDA(c, cudaMalloc(&c->d_gran_off, ((size_t)R + 1) * 4));
        PD_CUDA(c, cudaMalloc(&c->d_long_off, ((size_t)R + 1) * 4));
        c->cap_gran = need + need / 8;
    }
    PD_CUDA(c, cudaMemcpyAsync(c->d_gran_off, goff.data(), ((size_t)R + 1) * 4, cudaMemcpyHostToDevice, c->stream));
    PD_CUDA(c, cudaMemcpyAsync(c->d_long_off, c->h_long_off.data(), ((size_t)R + 1) * 4, cudaMemcpyHostToDevice, c->stream));
    PD_CUDA(c, cudaMemsetAsync(c->d_gran_tile, 0, need * 4, c->stream));
    pd_launch_gran_index(a, c->d_gran_tile, c->d_gran_off, c->stream);
    PD_CUDA(c, cudaGetLastError());
    PD_CUDA(c, cudaStreamSynchronize(c->stream));                    // goff (host vector) is read by the async copy
    c->index_built = true;
    return 0;
}

// device view of the uploaded contig (the window range and thresholds are the caller's); builds the index once per upload
int device_view(pd_ctx * c, PdDev & a)
{
    a = PdDev{};
    a.words = c->d_words; a.tiles = c->d_tiles; a.longs = c->d_longs;
    a.rgc = c->d_rgc; a.sample_rg = c->d_sample_rg; a.tab = c->d_tab;
    a.NT = c->NT; a.N = c->N; a.R = c->R; a.window_buffer = c->grid.window_buffer; a.t_min = c->t_min;
    a.tseg = c->d_tseg;
    return c->index_built ? 0 : build_index(c, a);
}

// mapped, page-locked result buffers: grown so that `need_calls` calls fit; existing contents are preserved
int ensure_results(pd_ctx * c, size_t need_calls, size_t row, size_t keep_calls)
{
    if (!c->res_count) {
        PD_CUDA(c, cudaHostAlloc(&c->res_count, 256, cudaHostAllocMapped));      // [0] calls emitted; [16..31] counter read-back
        c->res_count[0] = 0;
    }
    if (need_calls > c->cap_res_calls || !c->res_calls) {
        const size_t want = std::max<size_t>(need_calls + need_calls / 2, 1024);
        pd_call * p = nullptr;
        PD_CUDA(c, cudaHostAlloc(&p, want * sizeof(pd_call), cudaHostAllocMapped));
        if (keep_calls) memcpy(p, c->res_calls, keep_calls * sizeof(pd_call));
        if (c->res_calls) cudaFreeHost(c->res_calls);
        c->res_calls = p; c->cap_res_calls = want;
    }
    if (need_calls * row > c->cap_res_ps || !c->res_ps) {
        const size_t want = std::max<size_t>((need_calls + need_calls / 2) * row, 1u << 18);
        uint32_t * p = nullptr;
        if (cudaHostAlloc(&p, want * 4, cudaHostAllocMapped) != cudaSuccess) {
            cudaGetLastError();
            return pd_fail(c, PD_ERR_CAPACITY, "cannot page-lock the result buffer for this many calls x samples; scan a smaller window range");
        }
        if (keep_calls) memcpy(p, c->res_ps, keep_calls * row * 4);
        if (c->res_ps) cudaFreeHost(c->res_ps);
        c->res_ps = p; c->cap_res_ps = want;
    }
    return 0;
}

// Samples of the cohort rounded up to a multiple of 32 (k_candidates' shared-memory row of Q3s and its block size)
uint32_t cand_npad(uint32_t n_global) { return (std::max<uint32_t>(n_global, 32) + 31u) & ~31u; }

// The instance of k_candidates that reads the Q3s from global memory: for cohorts whose Q3s do not fit its shared memory,
// or at any size with PD_CAND_GLOBAL=1 (tests: both instances on the same input)
bool cand_global(uint32_t npad)
{
    const char * e = getenv("PD_CAND_GLOBAL");
    return (size_t)npad * 4 > PD_CAND_SMEM || (e && atoi(e) != 0);
}

}  // namespace

int pd_run_scan(pd_ctx * c, uint64_t first_window, uint64_t n_windows, pd_result * out)
{
    PD_CUDA(c, cudaSetDevice(c->device));
    memset(out, 0, sizeof(*out));
    PdShard * sh = c->shard;                                          // sample-sharded cohort: this scan is a collective
    uint64_t total = c->n_windows_total;
    if (sh) {
        if (pd_shard_window_total(c, &total)) return c->status;
        if ((total + PD_TILE_WINDOWS - 1) / PD_TILE_WINDOWS > c->NT)
            return pd_fail(c, PD_ERR_ARG, "sample-sharded scan: the cohort's window range exceeds this rank's tile tables; call pd_contig_reserve_windows(contig length / 30 + 2) before the upload");
    }
    const uint64_t w_begin = std::min<uint64_t>(first_window, total);
    const uint64_t w_end = n_windows ? std::min<uint64_t>(first_window + n_windows, total) : total;
    const uint32_t N = c->N, R = c->R;
    // sizes that decide the batching must be the same on every rank of a sharded cohort
    const uint32_t Nb = sh ? sh->n_local_max : N, Rb = sh ? sh->r_global : R, Ng = sh ? sh->n_global : N;
    const size_t row = 13ull * N;
    const bool uni = c->unify_on;                                     // window calls stay on the device, merged there
    if (ensure_results(c, 1, row, 0)) return c->status;
    if (uni && pd_unify_ensure_raw(c, 1, row, 0)) return c->status;
    c->res_count[0] = 0;
    out->n_reads = c->n_reads;
    out->algorithmic_bytes = 4ull * c->n_reads;
    out->h2d_bytes = c->h2d_bytes;
    out->calls = c->res_calls; out->per_sample = c->res_ps;
    if (w_end <= w_begin) return 0;
    const uint32_t W = (uint32_t)(w_end - w_begin);
    out->n_windows = W;

    PdDev a;
    if (device_view(c, a)) return c->status;
    // Second screen stage (pd_gather.cu, k_screen2): worth it when the read groups have different initial-length thresholds,
    // i.e. when the cohort-minimum threshold t_min lets nearly every window through the first stage. PD_SCREEN2=0/1 overrides.
    bool screen2 = false;
    if (!sh) {
        uint32_t tmax = 0;
        for (const auto & k : c->rgc) tmax = std::max(tmax, k.min_init);
        screen2 = (int64_t)tmax > (int64_t)c->t_min && c->t_min >= 60;
        if (getenv("PD_SCREEN2")) screen2 = atoi(getenv("PD_SCREEN2")) != 0 && c->t_min >= 60;
    }
    const int s2gap = getenv("PD_SCREEN2_GAP") ? atoi(getenv("PD_SCREEN2_GAP")) : 30;     // (tuning knob)
    a.t_known = screen2 ? std::max(c->t_min - s2gap, c->t_min / 2) : 0;
    a.t_mark = screen2 ? a.t_known : a.t_min;
    a.w_begin = (uint32_t)w_begin; a.w_end = (uint32_t)w_end;

    cudaStream_t st = c->stream, st2 = c->stream2;
    uint64_t * nl = &out->n_kernel_launches;
    const bool dbg = getenv("PD_DEBUG") != nullptr;
    const int dbg_window = getenv("PD_DEBUG_WINDOW") ? atoi(getenv("PD_DEBUG_WINDOW")) : -1;

    // ---- screen
    ScreenArgs s;
    s.tile_begin = (uint32_t)(w_begin / PD_TILE_WINDOWS);
    s.tile_end = (uint32_t)std::min<uint64_t>((w_end + PD_TILE_WINDOWS - 1) / PD_TILE_WINDOWS, c->NT);
    s.tb_al = s.tile_begin & ~31u;
    s.need_stride = (s.tile_end - s.tb_al + 31) / 32;
    s.gran_off = c->d_gran_off; s.gran_tile = c->d_gran_tile; s.long_off = c->d_long_off;
    s.total_longs = (uint32_t)c->total_longs;
    const uint32_t n_tiles = s.tile_end - s.tile_begin;
    uint32_t * d_counters; unsigned long long * d_bsums;
    if (grow_scratch(c, S_NEED, s.need, (size_t)N * s.need_stride)) return c->status;
    if (grow_scratch(c, S_TFLAGS, s.tile_flags, (size_t)n_tiles)) return c->status;
    s.known = nullptr; s.kjobs = nullptr; s.kjobs_cap = 0; s.counters = nullptr;
    const size_t known_stride = (size_t)s.need_stride * 32;
    if (screen2) {
        if (grow_scratch(c, S_KNOWN, s.known, (size_t)N * known_stride)) return c->status;
        PD_CUDA(c, cudaMemsetAsync(s.known, 0, (size_t)N * known_stride * 4, st));
        const size_t kcap = std::min<size_t>((size_t)N * n_tiles, 0xFFFFFFF0ull);
        if (grow_scratch(c, S_KJOBS, s.kjobs, kcap)) return c->status;
        s.kjobs_cap = (uint32_t)kcap;
    }
    if (grow_scratch(c, S_COUNTERS, d_counters, (size_t)CNT_N)) return c->status;
    s.counters = d_counters;
    JobArgs j;
    j.tj_of_tile = nullptr;
    if (screen2) {
        if (grow_scratch(c, S_TJ_OF_TILE, j.tj_of_tile, (size_t)n_tiles)) return c->status;
        PD_CUDA(c, cudaMemsetAsync(j.tj_of_tile, 0xFF, (size_t)n_tiles * 4, st));
    }
    j.tile_flags = s.tile_flags; j.n_tiles = n_tiles; j.tile_begin = s.tile_begin; j.counters = d_counters;
    if (grow_scratch(c, S_TJ_TILE, j.tj_tile, (size_t)n_tiles)) return c->status;
    if (grow_scratch(c, S_TJ_MASK, j.tj_mask, (size_t)n_tiles)) return c->status;
    if (grow_scratch(c, S_TJ_WBASE, j.tj_wbase, (size_t)n_tiles)) return c->status;
    if (grow_scratch(c, S_JOBWIN, j.job_window, (size_t)n_tiles * PD_TILE_WINDOWS)) return c->status;
    if (grow_scratch(c, S_BSUMS, d_bsums, (size_t)std::max<uint64_t>((n_tiles * (uint64_t)PD_TILE_WINDOWS + 1023) / 1024, 1) + 1)) return c->status;
    j.block_sums = d_bsums;
    PD_CUDA(c, cudaEventRecord(c->ev[2], st));
    PD_CUDA(c, cudaMemsetAsync(s.need, 0, (size_t)N * s.need_stride * 4, st));
    PD_CUDA(c, cudaMemsetAsync(s.tile_flags, 0, (size_t)n_tiles * 4, st));
    PD_CUDA(c, cudaMemsetAsync(d_counters, 0, CNT_N * 4, st));
    PD_CUDA(c, cudaEventRecord(c->ev[3], st));
    if (n_tiles) {
        pd_launch_screen(a, s, c->max_rg_words, st, c->ev[10], nl);
        PD_CUDA(c, cudaGetLastError());
    }
    if (sh && n_tiles && pd_shard_or_flags(c, s.tile_flags, n_tiles, st)) return c->status;      // a window is flagged if ANY rank flags it
    PD_CUDA(c, cudaEventRecord(c->ev[4], st));
    if (n_tiles) pd_launch_tile_jobs(j, st, nl);
    PD_CUDA(c, cudaGetLastError());
    uint32_t * h_cnt = c->res_count + 16;                            // page-locked: the read-back is a plain DMA
    PD_CUDA(c, cudaMemcpyAsync(h_cnt, d_counters, CNT_N * 4, cudaMemcpyDeviceToHost, st));
    PD_CUDA(c, cudaStreamSynchronize(st));
    const uint32_t n_tj = h_cnt[CNT_TJOBS], n_jobs = h_cnt[CNT_JOBS];
    out->n_flagged_windows = n_jobs;

    // ---- genotyping stage. Level 1: batches of tile jobs (Q3 of every flagged window, candidates). Level 2: the windows
    // with candidates ("candidate jobs") in sub-batches of whole tiles (active-set pool, EM, final pass, emission).
    const uint32_t npad = cand_npad(Ng);
    const bool cglobal = cand_global(npad);
    const size_t job_bytes = 9ull * Nb * (sh ? sh->world + 1 : 1) + (cglobal ? 4ull * npad : 0) + 4ull * (PD_CAND_INLINE + 3) + 8;
    uint32_t JB = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(3000000000ull / job_bytes, 64), 1u << 20);
    if (getenv("PD_JOB_BATCH")) JB = std::max<uint32_t>((uint32_t)atoi(getenv("PD_JOB_BATCH")), 64);           // test knobs
    const uint32_t rows_env = getenv("PD_CJOB_ROWS") ? std::max<uint32_t>((uint32_t)atoi(getenv("PD_CJOB_ROWS")), 1) : 0;
    const uint32_t slow_env = getenv("PD_FORCE_SLOW") ? (uint32_t)atoi(getenv("PD_FORCE_SLOW")) : 0;
    const size_t cjob_bytes = 8ull * Rb + 400ull * Nb;
    const uint32_t JB2 = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(4000000000ull / cjob_bytes, 64), 1u << 20);
    std::vector<uint32_t> h_wbase;
    if (n_jobs > JB) {
        h_wbase.resize(n_tj);
        PD_CUDA(c, cudaMemcpyAsync(h_wbase.data(), j.tj_wbase, (size_t)n_tj * 4, cudaMemcpyDeviceToHost, st));
        PD_CUDA(c, cudaStreamSynchronize(st));
    }
    const bool em2 = !sh && pd_em2_usable(c);                          // sample-major pipeline (pd_em2.cu)
    // (reads per pair are not known before the gather: budget 40 active read pairs per read group)
    const size_t pair_bytes = 48ull * Nb + 4ull * Rb + 2 * 52ull * Nb + 128 + (em2 ? pd_em2_pair_bytes(Rb, 40.0 * Rb) : 0);
    const uint32_t CH = (uint32_t)std::min<uint64_t>(std::max<uint64_t>((em2 ? 6000000000ull : 2000000000ull) / pair_bytes, 64),
                                                     getenv("PD_EM_CHUNK") ? atoi(getenv("PD_EM_CHUNK")) : 16384);
    // (measured on B200, 100 samples x chr21: tapering costs more in small EM launches than it saves in the tail -> off by default)
    const uint32_t taper_min = std::min<uint32_t>(CH, getenv("PD_EM_TAPER") ? std::max(1, atoi(getenv("PD_EM_TAPER"))) : CH);
    XrArgs xr;
    memset(&xr, 0, sizeof(xr));
    if (sh) {
        xr.world = sh->world; xr.rank = sh->rank; xr.pairs_cap = sh->xr_pairs_cap; xr.ticket = sh->d_ticket; xr.err = sh->d_err;
        xr.n_global = sh->n_global; xr.owns_rg0 = sh->sample_offset == 0; xr.grid_cap = sh->grid_cap;
        for (uint32_t r = 0; r < sh->world; ++r) xr.peer[r] = sh->xr_peer[r];
        if (CH > sh->xr_pairs_cap) return pd_fail(c, PD_ERR_ARG, "EM chunk larger than the exchange slots");
        PD_CUDA(c, cudaMemsetAsync(sh->d_err, 0, 4, st));
    }
    uint64_t n_pairs_total = 0, n_cjobs_total = 0;
    uint32_t chunk_no = 0;
    std::vector<uint32_t> h_jobwin; std::vector<PdPair> h_pairs;
    std::vector<uint32_t> h_cfirst, h_cmask, h_tjw, h_cand_off;
    if (dbg && n_jobs) {
        h_jobwin.resize(n_jobs);
        PD_CUDA(c, cudaMemcpy(h_jobwin.data(), j.job_window, (size_t)n_jobs * 4, cudaMemcpyDeviceToHost));
    }
    uint32_t * d_emit_state;
    if (grow_scratch(c, S_CHUNK_BASE, d_emit_state, (size_t)4)) return c->status;
    PD_CUDA(c, cudaMemsetAsync(d_emit_state, 0, 16, st));
    if (em2) {
        uint32_t * e2cnt;
        if (grow_scratch(c, PD_S_E2_CNT, e2cnt, (size_t)8)) return c->status;
        PD_CUDA(c, cudaMemsetAsync(e2cnt, 0, 32, st));
    }
    double pool_words_last = 0;                                       // read pairs in the pool of the current sub-batch

    for (uint32_t tj0 = 0; tj0 < n_tj;) {
        // batch = tile jobs [tj0, tj1) with at most JB window jobs
        uint32_t tj1 = n_tj, job_base = 0, nj = n_jobs;
        if (!h_wbase.empty()) {
            job_base = h_wbase[tj0];
            tj1 = tj0 + 1;
            while (tj1 < n_tj && h_wbase[tj1] - job_base <= JB - PD_TILE_WINDOWS) ++tj1;
            nj = (tj1 < n_tj ? h_wbase[tj1] : n_jobs) - job_base;
        }
        const uint32_t ntj = tj1 - tj0;
        GatherArgs ga;
        memset(&ga, 0, sizeof(ga));
        ga.tj_tile = j.tj_tile; ga.tj_mask = j.tj_mask; ga.tj_wbase = j.tj_wbase; ga.tj0 = tj0; ga.ntj = ntj;
        ga.job_base = job_base; ga.counters = d_counters;
        if (grow_scratch(c, S_Q3, ga.q3, (size_t)nj * Nb)) return c->status;         // (sharded: all-gather blocks of equal size)
        if (grow_scratch(c, S_SSTAT, ga.sstat, (size_t)nj * Nb)) return c->status;
        if (grow_scratch(c, S_DMAX, ga.dmax, (size_t)nj * N)) return c->status;
        uint32_t * d_cmask, * d_cfirst;
        if (grow_scratch(c, S_TJ_CMASK, d_cmask, (size_t)ntj)) return c->status;
        if (grow_scratch(c, S_TJ_CFIRST, d_cfirst, (size_t)ntj)) return c->status;
        ga.tj_cmask = d_cmask; ga.tj_cfirst = d_cfirst;
        ga.phase = 0; ga.known = s.known; ga.known_stride = (uint32_t)known_stride; ga.tb_al = s.tb_al;
        ga.kjobs = s.kjobs; ga.n_kjobs = std::min<uint32_t>(h_cnt[CNT_KJOBS], s.kjobs_cap); ga.tj_of_tile = j.tj_of_tile; ga.tile_begin = s.tile_begin;
        if (screen2) {
            if (grow_scratch(c, S_TJ_ALIVE, ga.tj_alive, (size_t)ntj)) return c->status;
            if (grow_scratch(c, S_JOB_DEAD, ga.job_dead, (size_t)nj)) return c->status;
        }
        CandArgs ca;
        memset(&ca, 0, sizeof(ca));
        ca.nparts = 1; ca.q3[0] = ga.q3; ca.sstat[0] = ga.sstat; ca.part_n[0] = N; ca.min_init = c->d_min_init;
        ca.njobs = nj; ca.job_base = job_base; ca.counters = d_counters; ca.block_sums = d_bsums; ca.npad = npad;
        ca.force_sort = (slow_env >> 2) & 1u;
        if (cglobal && grow_scratch(c, S_CAND_SORT, ca.sort_buf, (size_t)nj * npad)) return c->status;
        ca.job_dead = screen2 ? ga.job_dead : nullptr;
        int32_t * all_q3 = nullptr; uint8_t * all_ss = nullptr;
        if (sh) {
            if (grow_scratch(c, S_ALL_Q3, all_q3, (size_t)nj * Nb * sh->world)) return c->status;
            if (grow_scratch(c, S_ALL_SS, all_ss, (size_t)nj * Nb * sh->world)) return c->status;
            ca.nparts = sh->world;
            for (uint32_t r = 0; r < sh->world; ++r) {
                ca.q3[r] = all_q3 + (size_t)r * nj * Nb; ca.sstat[r] = all_ss + (size_t)r * nj * Nb; ca.part_n[r] = sh->part_n[r];
            }
        }
        if (grow_scratch(c, S_CAND_CNT, ca.cand_cnt, (size_t)nj)) return c->status;
        if (grow_scratch(c, S_CAND_INL, ca.cand_inline, (size_t)nj * PD_CAND_INLINE)) return c->status;
        if (grow_scratch(c, S_CAND_OFF, ca.cand_off, (size_t)nj)) return c->status;
        if (grow_scratch(c, S_CJOB_OF, ca.cjob_of, (size_t)nj)) return c->status;
        uint32_t rows_cap = std::min<uint32_t>(std::min<uint32_t>(nj, JB2), (uint32_t)std::max<uint64_t>(1000000000ull / (8ull * Rb), 64));
        if (rows_env) rows_cap = std::min(rows_cap, rows_env);
        ga.debug_flags = slow_env;
        if (grow_scratch(c, S_ACT_OFF, ga.act_off, (size_t)(rows_cap + PD_TILE_WINDOWS) * R)) return c->status;
        if (grow_scratch(c, S_ACT_CNT, ga.act_cnt, (size_t)(rows_cap + PD_TILE_WINDOWS) * R)) return c->status;
        size_t pair_cap = std::max<size_t>(c->cap_scratch[S_PAIRS] / sizeof(PdPair), (size_t)nj * 2 + 1024);
        if (c->pool_cap == 0) c->pool_cap = std::max<size_t>((size_t)std::min<uint32_t>(nj, 16384) * R * 40, 1u << 20);

        if (screen2) {
            ga.phase = 1; pd_launch_q3(a, ga, st, nl);               // exact Q3 of the (window, sample) pairs that can exceed t_known
            pd_launch_screen2(a, ga, st, nl);                        // windows without a possible candidate drop out
            ga.phase = 2; pd_launch_q3(a, ga, st, nl);               // the rest of the surviving windows
            ga.phase = 0;
        } else pd_launch_q3(a, ga, st, nl);
        PD_CUDA(c, cudaGetLastError());
        if (sh) {                                                   // every rank derives the candidates from ALL samples' Q3
            if (pd_shard_allgather(c, ga.q3, all_q3, (size_t)nj * Nb * 4, st)) return c->status;
            if (pd_shard_allgather(c, ga.sstat, all_ss, (size_t)nj * Nb, st)) return c->status;
        }
        // candidates, then (optimistically) the pool of the first sub-batch; one synchronisation validates both
        auto run_gather = [&](uint32_t cj_lo) -> int {
            if (c->pool_cap > 0xFFFFFFF0ull) c->pool_cap = 0xFFFFFFF0ull;
            if (grow_scratch(c, S_POOL_POS, ga.pool_pos, c->pool_cap)) return c->status;
            if (grow_scratch(c, S_POOL_DEV, ga.pool_dev, c->pool_cap)) return c->status;
            ga.pool_cap = (uint32_t)c->pool_cap; ga.cj_base = cj_lo; ga.cj_end = cj_lo + rows_cap;
            PD_CUDA(c, cudaMemsetAsync(d_counters + CNT_POOL, 0, 4, st));
            pd_launch_gather(a, ga, st, nl);
            PD_CUDA(c, cudaGetLastError());
            return 0;
        };
        uint32_t n_pairs = 0, n_cj = 0;
        bool cand_done = false;
        for (int attempt = 0; ; ++attempt) {
            if (grow_scratch(c, S_PAIRS, ca.pairs, pair_cap)) return c->status;
            ca.pair_cap = (uint32_t)std::min<size_t>(pair_cap, 0xFFFFFFF0ull);
            if (!cand_done) {
                if (pd_launch_candidates(c, a, ca, st, nl)) return c->status;
                pd_launch_cmask(ga, ca, d_cmask, d_cfirst, st, nl);
            }
            if (run_gather(0)) return c->status;
            PD_CUDA(c, cudaMemcpyAsync(h_cnt, d_counters, CNT_N * 4, cudaMemcpyDeviceToHost, st));
            PD_CUDA(c, cudaStreamSynchronize(st));
            const bool pool_ok = h_cnt[CNT_POOL] <= c->pool_cap, pairs_ok = h_cnt[CNT_PAIRS] <= pair_cap;
            if (pool_ok && pairs_ok) { n_pairs = h_cnt[CNT_PAIRS]; n_cj = h_cnt[CNT_CJOBS]; pool_words_last = h_cnt[CNT_POOL]; break; }
            if (attempt == 3) return pd_fail(c, PD_ERR_CAPACITY, "active read-pair pool / candidate list overflow");
            if (!pool_ok) c->pool_cap = (size_t)h_cnt[CNT_POOL] + (size_t)h_cnt[CNT_POOL] / 8 + 1024;      // exact size known now: run again
            if (pairs_ok) cand_done = true;
            else pair_cap = (size_t)h_cnt[CNT_PAIRS] + 1024;
        }
        n_pairs_total += n_pairs; n_cjobs_total += n_cj;
        if (dbg && n_pairs) {
            h_pairs.resize(n_pairs);
            PD_CUDA(c, cudaMemcpy(h_pairs.data(), ca.pairs, (size_t)n_pairs * sizeof(PdPair), cudaMemcpyDeviceToHost));
        }
        const bool multi = n_cj > rows_cap;
        if (multi) {                    // sub-batch borders need the tiles' candidate-job numbering on the host
            h_cfirst.resize(ntj); h_cmask.resize(ntj); h_tjw.resize(ntj); h_cand_off.resize(nj);
            PD_CUDA(c, cudaMemcpyAsync(h_cfirst.data(), d_cfirst, (size_t)ntj * 4, cudaMemcpyDeviceToHost, st));
            PD_CUDA(c, cudaMemcpyAsync(h_cmask.data(), d_cmask, (size_t)ntj * 4, cudaMemcpyDeviceToHost, st));
            PD_CUDA(c, cudaMemcpyAsync(h_tjw.data(), j.tj_wbase + tj0, (size_t)ntj * 4, cudaMemcpyDeviceToHost, st));
            PD_CUDA(c, cudaMemcpyAsync(h_cand_off.data(), ca.cand_off, (size_t)nj * 4, cudaMemcpyDeviceToHost, st));
            PD_CUDA(c, cudaStreamSynchronize(st));
        }
        // first pair of the first tile whose first candidate job is >= cj
        auto pair_at = [&](uint32_t cj) -> uint32_t {
            for (uint32_t t = 0; t < ntj; ++t)           // (sub-batches are few; a linear scan is fine)
                if (h_cmask[t] && h_cfirst[t] >= cj) return h_cand_off[h_tjw[t] - job_base];
            return n_pairs;
        };

        for (uint32_t cj_lo = 0; cj_lo < std::max<uint32_t>(n_cj, 1) && n_pairs; cj_lo += rows_cap) {
            uint32_t pA = 0, pB = n_pairs;
            if (multi) {
                pA = pair_at(cj_lo); pB = pair_at(cj_lo + rows_cap);
                if (cj_lo > 0) {
                    for (int attempt = 0; ; ++attempt) {
                        if (run_gather(cj_lo)) return c->status;
                        PD_CUDA(c, cudaMemcpyAsync(h_cnt, d_counters, CNT_N * 4, cudaMemcpyDeviceToHost, st));
                        PD_CUDA(c, cudaStreamSynchronize(st));
                        if (h_cnt[CNT_POOL] <= c->pool_cap) { pool_words_last = h_cnt[CNT_POOL]; break; }
                        if (attempt == 2) return pd_fail(c, PD_ERR_CAPACITY, "active read-pair pool overflow");
                        c->pool_cap = (size_t)h_cnt[CNT_POOL] + (size_t)h_cnt[CNT_POOL] / 8 + 1024;
                    }
                }
            }
            // ---- pairs in chunks: the emission of chunk k (stream2) overlaps the EM of chunk k+1 (stream)
            // Optional (PD_EM_TAPER): chunk sizes taper off (3/4 of what is left) so that the emission of the LAST chunk,
            // which no EM launch hides, is small. Deterministic in (pairs, CH): identical on every rank.
            for (uint32_t p0 = pA, np = 0; p0 < pB; p0 += np, ++chunk_no) {
                const uint32_t left = pB - p0;
                np = std::min(CH, left <= taper_min + taper_min / 2 ? left : std::max(taper_min, (uint32_t)((uint64_t)left * 3 / 4 / taper_min * taper_min)));
                const int par = (int)(chunk_no & 1);
                EmArgs e;
                if (grow_scratch(c, S_DLX, e.dlx, (size_t)CH * 3 * N)) return c->status;
                if (grow_scratch(c, S_DLE, e.dle, (size_t)CH * 3 * N)) return c->status;
                if (grow_scratch(c, S_SHIFTS, e.shifts, (size_t)CH * R)) return c->status;
                if (grow_scratch(c, S_STATES, e.states, (size_t)CH)) return c->status;
                // double-buffered: read by stream2 while the next chunk is computed
                if (chunk_no >= 2) PD_CUDA(c, cudaStreamWaitEvent(st, c->ev[8 + par], 0));          // chunk k-2 has been emitted
                if (grow_scratch(c, S_PS0 + par, e.ps, (size_t)CH * row)) return c->status;
                if (grow_scratch(c, S_CALLS0 + par, e.calls, (size_t)CH)) return c->status;
                if (grow_scratch(c, S_VALID0 + par, e.valid, (size_t)CH + 16)) return c->status;
                if (grow_scratch(c, S_DONE0 + par, e.done, (size_t)CH)) return c->status;
                e.job_window = j.job_window; e.pairs = ca.pairs; e.pair0 = p0; e.npairs = np; e.job_base = job_base;
                e.pool_pos = ga.pool_pos; e.pool_dev = ga.pool_dev; e.act_off = ga.act_off; e.act_cnt = ga.act_cnt; e.sstat = ga.sstat; e.dmax = ga.dmax;
                e.cjob_of = ca.cjob_of; e.cj_base = cj_lo;
                e.xr = xr;
                if (sh) e.xr.epoch = sh->epoch++;
                e.iterations = c->params.iterations; e.min_len = c->params.min_len; e.min_lr = c->params.min_lr;
                e.min_sample_fraction = c->params.min_sample_fraction; e.somatic = c->params.somatic; e.window_wise = c->params.window_wise;
                e.anchor = c->grid.anchor;
                e.dbg = nullptr; e.dbg_window = dbg_window;
                e.sort_samples = getenv("PD_EM_SORT") ? atoi(getenv("PD_EM_SORT")) : 1;
                if (dbg) {
                    if (grow_scratch(c, S_DBG, e.dbg, (size_t)CH * 4)) return c->status;
                    PD_CUDA(c, cudaMemsetAsync(e.dbg, 0xFF, (size_t)np * 16, st));
                }
                PD_CUDA(c, cudaMemsetAsync(e.valid, 0, np, st));
                PD_CUDA(c, cudaMemsetAsync(e.done, 0, (size_t)np * 4, st));
                // result capacity: upper bound = calls emitted so far (exact once stream2 is drained) + this chunk
                const size_t upper = (size_t)(n_pairs_total - n_pairs + p0 + np);
                if (uni ? (upper > c->cap_u_calls || upper * row > c->cap_u_ps) : (upper > c->cap_res_calls || upper * row > c->cap_res_ps)) {
                    PD_CUDA(c, cudaStreamSynchronize(st2));
                    const size_t have = c->res_count[0];
                    if (uni ? pd_unify_ensure_raw(c, have + np, row, have) : ensure_results(c, have + np, row, have)) return c->status;
                }
                // the emitter of this chunk starts on stream2 as soon as the flags are cleared and runs CONCURRENTLY with
                // the EM launch below, copying finished pairs to the host in pair order while later pairs are computed
                PD_CUDA(c, cudaEventRecord(c->ev[6 + par], st));
                EmitArgs m;
                m.valid = e.valid; m.calls = e.calls; m.ps = e.ps; m.npairs = np; m.row_words = (uint32_t)row; m.done = e.done;
                m.counters = d_counters; m.emit_blocks_done = d_emit_state;
                m.out_calls = uni ? c->d_u_calls : c->res_calls; m.out_ps = uni ? c->d_u_ps : c->res_ps; m.out_count = c->res_count;
                if (sh && pd_shard_prelaunch(c)) return c->status;
                // (EM first: CUDA loads kernels lazily and a first-time load may wait for running kernels -- the emitter,
                // which only waits for ev[6], must never be the one that is running while the EM kernel is being loaded)
                const bool time_em = chunk_no == 0;
                if (time_em) PD_CUDA(c, cudaEventRecord(c->ev[12], st));
                if (em2) {
                    const uint32_t rows_here = std::max<uint32_t>(std::min<uint32_t>(n_cj - std::min(n_cj, cj_lo), rows_cap), 1);
                    if (pd_launch_em2(c, a, e, pool_words_last / rows_here, st, nl)) return c->status;
                    PD_CUDA(c, cudaEventRecord(c->ev[6 + par], st));            // the emitter starts when the chunk is complete
                } else if (pd_launch_em(c, a, e, st, nl)) return c->status;
                if (time_em) { PD_CUDA(c, cudaEventRecord(c->ev[13], st)); out->n_em_pairs_timed = np; }
                PD_CUDA(c, cudaStreamWaitEvent(st2, c->ev[6 + par], 0));
                pd_launch_emit(m, st2, nl);
                PD_CUDA(c, cudaGetLastError());
                PD_CUDA(c, cudaEventRecord(c->ev[8 + par], st2));
                if (dbg) {
                    std::vector<uint32_t> hd((size_t)np * 4);
                    PD_CUDA(c, cudaMemcpyAsync(hd.data(), e.dbg, (size_t)np * 16, cudaMemcpyDeviceToHost, st));
                    PD_CUDA(c, cudaStreamSynchronize(st));
                    for (uint32_t i = 0; i < np; ++i)
                        fprintf(stderr, "PD_DEBUG pair window %u L0 %d reason %u len %u it %u supp %u\n", h_jobwin[h_pairs[p0 + i].job],
                                h_pairs[p0 + i].L0, hd[4 * i], hd[4 * i + 1], hd[4 * i + 2], hd[4 * i + 3]);
                }
            }
        }
        // the next batch overwrites the Q3 / pool / active-set tables that the EM kernels of this batch read: stream
        // order on `stream` covers that; the pair list is only read by the EM kernels as well.
        tj0 = tj1;
    }
    PD_CUDA(c, cudaEventRecord(c->ev[5], st));
    PD_CUDA(c, cudaStreamSynchronize(st));
    PD_CUDA(c, cudaStreamSynchronize(st2));
    PD_CUDA(c, cudaMemcpy(h_cnt, d_counters, CNT_N * 4, cudaMemcpyDeviceToHost));
    if (em2) {
        bool ovf = false; size_t need = 0;
        if (pd_em2_overflow(c, &ovf, &need)) return c->status;
        if (ovf) {                                                    // the interleaved read-pair copies did not fit: once more with room
            if (c->e2_retry >= 4) return pd_fail(c, PD_ERR_CAPACITY, "EM read-pair copies overflow");
            ++c->e2_retry;
            c->e2_devt_cap = std::max<size_t>(c->e2_devt_cap * 2, need + need / 4);
            const int rc = pd_run_scan(c, first_window, n_windows, out);
            --c->e2_retry;
            return rc;
        }
    }
    if (h_cnt[CNT_ERR]) return pd_fail(c, PD_ERR_CUDA, "the result emitter gave up waiting for the EM kernels");
    if (sh) {
        uint32_t xerr = 0;
        PD_CUDA(c, cudaMemcpy(&xerr, sh->d_err, 4, cudaMemcpyDeviceToHost));
        if (xerr) return pd_fail(c, PD_ERR_CUDA, "sample-sharded scan: a peer rank did not answer an in-kernel exchange in time");
    }
    out->n_calls = c->res_count[0];
    out->n_window_calls = out->n_calls;
    out->n_screened_windows = screen2 ? h_cnt[CNT_ALIVE] : out->n_flagged_windows;
    out->n_known_pairs = screen2 ? h_cnt[CNT_KNOWN] : 0;
    if (out->n_em_pairs_timed) PD_CUDA(c, cudaEventElapsedTime(&out->ms_em, c->ev[12], c->ev[13]));
    if (uni) {
        const uint32_t nseg = (uint32_t)((w_end * PD_WIN) / c->grid.window_buffer + 2);
        PD_CUDA(c, cudaEventRecord(c->ev[11], st));
        if (pd_run_unify(c, (uint32_t)out->n_window_calls, row, nseg, ensure_results, &out->n_calls, nl)) return c->status;
        PD_CUDA(c, cudaEventRecord(c->ev[5], st));
        PD_CUDA(c, cudaStreamSynchronize(st));
        PD_CUDA(c, cudaEventElapsedTime(&out->ms_unify, c->ev[11], c->ev[5]));
        out->significant_windows = c->res_sig;
    }
    out->calls = c->res_calls;
    out->per_sample = c->res_ps;
    out->n_candidates = n_pairs_total;
    out->d2h_bytes = out->n_calls * (sizeof(pd_call) + row * 4);
    PD_CUDA(c, cudaEventElapsedTime(&out->ms_screen, c->ev[3], c->ev[4]));
    if (n_tiles) PD_CUDA(c, cudaEventElapsedTime(&out->ms_stream, c->ev[3], c->ev[10]));
    PD_CUDA(c, cudaEventElapsedTime(&out->ms_genotype, c->ev[4], c->ev[5]));
    PD_CUDA(c, cudaEventElapsedTime(&out->ms_total, c->ev[2], c->ev[5]));
    out->ms_d2h = 0;
    return 0;
}

// ---------------------------------------------------------------------------------------------------------
// device-side validation hook: per-window sums of one read group as the scan kernels' read-pair walk sees them
// ---------------------------------------------------------------------------------------------------------
extern "C" int pd_debug_device_window_sums(pd_ctx * c, uint32_t rg, uint64_t first_window, uint64_t n_windows, int64_t * out)
{
    if (!c || !out || rg >= c->R) return PD_ERR_ARG;
    if (c->status) return c->status;
    if (c->device < 0) return pd_fail(c, PD_ERR_CUDA, "pd_debug_device_window_sums: host-only context (device = -1)");
    if (!c->contig_open) return pd_fail(c, PD_ERR_ARG, "no open contig");
    if (!c->uploaded) { const int rc = pd_contig_upload(c); if (rc) return rc; }
    PD_CUDA(c, cudaSetDevice(c->device));
    PdDev a;
    if (device_view(c, a)) return c->status;
    memset(out, 0, sizeof(int64_t) * 3 * n_windows);
    const uint64_t t0 = first_window / PD_TILE_WINDOWS;
    const uint64_t t1 = std::min<uint64_t>((first_window + n_windows + PD_TILE_WINDOWS - 1) / PD_TILE_WINDOWS, c->NT);
    if (n_windows == 0 || t0 >= t1) return 0;
    unsigned long long * d_out = nullptr;
    const size_t bytes = sizeof(unsigned long long) * 3 * n_windows;
    PD_CUDA(c, cudaMalloc(&d_out, bytes));
    cudaError_t e = cudaMemsetAsync(d_out, 0, bytes, c->stream);
    if (e == cudaSuccess) {
        pd_launch_window_sums(a, rg, c->grid.anchor, (uint32_t)t0, (uint32_t)t1, first_window, first_window + n_windows, d_out, c->stream);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, bytes, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d_out);
    if (e != cudaSuccess) return pd_fail(c, PD_ERR_CUDA, std::string("pd_debug_device_window_sums: ") + cudaGetErrorString(e));
    return 0;
}

// ---------------------------------------------------------------------------------------------------------
// device-side validation hook: the segment-level merge (pd_run_unify) of caller-built window calls
// ---------------------------------------------------------------------------------------------------------
extern "C" int pd_debug_unify(pd_ctx * c, uint64_t n, const pd_call * calls, const uint32_t * per_sample, uint32_t nseg, pd_result * out)
{
    if (!c || !out || (n && (!calls || !per_sample))) return PD_ERR_ARG;
    if (c->status) return c->status;
    if (c->device < 0) return pd_fail(c, PD_ERR_ARG, "pd_debug_unify: host-only context (device = -1)");
    if (!c->unify_on) return pd_fail(c, PD_ERR_ARG, "pd_debug_unify: no unify settings (call pd_set_unify first)");
    if (c->shard) return pd_fail(c, PD_ERR_ARG, "pd_debug_unify: sample-sharded context (the probe merges one context's calls)");
    if (n > 0xFFFFFFFFull) return pd_fail(c, PD_ERR_ARG, "pd_debug_unify: more than 2^32 - 1 window calls");
    for (uint64_t i = 0; i < n; ++i)      // the merge takes a segment's calls as one run of equal tags (k_seg_bounds)
        if (calls[i].segment >= nseg || (i && calls[i].segment < calls[i - 1].segment))
            return pd_fail(c, PD_ERR_ARG, "pd_debug_unify: segment tags must be < nseg and in ascending order");
    PD_CUDA(c, cudaSetDevice(c->device));
    memset(out, 0, sizeof(*out));
    const size_t row = 13ull * c->N;
    if (ensure_results(c, 1, row, 0)) return c->status;
    if (pd_unify_ensure_raw(c, std::max<uint64_t>(n, 1), row, 0)) return c->status;
    if (n) {
        PD_CUDA(c, cudaMemcpyAsync(c->d_u_calls, calls, n * sizeof(pd_call), cudaMemcpyHostToDevice, c->stream));
        PD_CUDA(c, cudaMemcpyAsync(c->d_u_ps, per_sample, n * row * 4, cudaMemcpyHostToDevice, c->stream));
    }
    out->n_window_calls = n;
    if (pd_run_unify(c, (uint32_t)n, row, nseg, ensure_results, &out->n_calls, &out->n_kernel_launches)) return c->status;
    PD_CUDA(c, cudaStreamSynchronize(c->stream));
    out->calls = c->res_calls;
    out->per_sample = c->res_ps;
    out->significant_windows = c->res_sig;
    return 0;
}

// ---------------------------------------------------------------------------------------------------------
// device-side validation hook: the candidate step (pd_launch_candidates) on caller-built Q3 / state rows
// ---------------------------------------------------------------------------------------------------------
extern "C" int pd_debug_candidates(pd_ctx * c, uint64_t n_windows, const int32_t * q3, const uint8_t * state, uint32_t * counts,
                                   int32_t * cands, uint64_t cap)
{
    if (!c || (n_windows && (!q3 || !state || !counts)) || (cap && !cands)) return PD_ERR_ARG;
    if (c->status) return c->status;
    if (c->device < 0) return pd_fail(c, PD_ERR_ARG, "pd_debug_candidates: host-only context (device = -1)");
    if (c->shard) return pd_fail(c, PD_ERR_ARG, "pd_debug_candidates: sample-sharded context (the probe takes one context's Q3 rows)");
    if (n_windows > 0x7FFFFFFFull) return pd_fail(c, PD_ERR_ARG, "pd_debug_candidates: more than 2^31 - 1 windows");
    if (n_windows == 0) return 0;
    PD_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const uint32_t nj = (uint32_t)n_windows, N = c->N, npad = cand_npad(N);
    PdDev a{};
    a.N = N; a.R = c->R; a.t_min = c->t_min;
    CandArgs ca;
    memset(&ca, 0, sizeof(ca));
    int32_t * d_q3; uint8_t * d_ss;
    if (grow_scratch(c, S_Q3, d_q3, (size_t)nj * N)) return c->status;
    if (grow_scratch(c, S_SSTAT, d_ss, (size_t)nj * N)) return c->status;
    PD_CUDA(c, cudaMemcpyAsync(d_q3, q3, (size_t)nj * N * 4, cudaMemcpyHostToDevice, st));
    PD_CUDA(c, cudaMemcpyAsync(d_ss, state, (size_t)nj * N, cudaMemcpyHostToDevice, st));
    ca.nparts = 1; ca.q3[0] = d_q3; ca.sstat[0] = d_ss; ca.part_n[0] = N; ca.min_init = c->d_min_init;
    ca.njobs = nj; ca.job_base = 0; ca.npad = npad;
    ca.force_sort = ((getenv("PD_FORCE_SLOW") ? (uint32_t)atoi(getenv("PD_FORCE_SLOW")) : 0u) >> 2) & 1u;
    if (cand_global(npad) && grow_scratch(c, S_CAND_SORT, ca.sort_buf, (size_t)nj * npad)) return c->status;
    if (grow_scratch(c, S_COUNTERS, ca.counters, (size_t)CNT_N)) return c->status;
    if (grow_scratch(c, S_BSUMS, ca.block_sums, (size_t)(nj + 1023) / 1024 + 1)) return c->status;
    if (grow_scratch(c, S_CAND_CNT, ca.cand_cnt, (size_t)nj)) return c->status;
    if (grow_scratch(c, S_CAND_INL, ca.cand_inline, (size_t)nj * PD_CAND_INLINE)) return c->status;
    if (grow_scratch(c, S_CAND_OFF, ca.cand_off, (size_t)nj)) return c->status;
    if (grow_scratch(c, S_CJOB_OF, ca.cjob_of, (size_t)nj)) return c->status;
    size_t pair_cap = std::max<size_t>(c->cap_scratch[S_PAIRS] / sizeof(PdPair), (size_t)nj * 2 + 1024);
    uint32_t cnt[CNT_N];
    uint64_t launches = 0;
    for (int attempt = 0; ; ++attempt) {                              // (a second attempt has the exact size)
        if (grow_scratch(c, S_PAIRS, ca.pairs, pair_cap)) return c->status;
        ca.pair_cap = (uint32_t)std::min<size_t>(pair_cap, 0xFFFFFFF0ull);
        if (pd_launch_candidates(c, a, ca, st, &launches)) return c->status;
        PD_CUDA(c, cudaMemcpyAsync(cnt, ca.counters, sizeof(cnt), cudaMemcpyDeviceToHost, st));
        PD_CUDA(c, cudaStreamSynchronize(st));
        if (cnt[CNT_PAIRS] <= ca.pair_cap) break;
        if (attempt == 1) return pd_fail(c, PD_ERR_CAPACITY, "pd_debug_candidates: candidate list overflow");
        pair_cap = (size_t)cnt[CNT_PAIRS] + 1024;
    }
    const uint32_t total = cnt[CNT_PAIRS];
    std::vector<PdPair> pairs(total);
    PD_CUDA(c, cudaMemcpyAsync(counts, ca.cand_cnt, (size_t)nj * 4, cudaMemcpyDeviceToHost, st));
    if (total) PD_CUDA(c, cudaMemcpyAsync(pairs.data(), ca.pairs, (size_t)total * sizeof(PdPair), cudaMemcpyDeviceToHost, st));
    PD_CUDA(c, cudaStreamSynchronize(st));
    for (uint64_t i = 0; i < std::min<uint64_t>(total, cap); ++i) cands[i] = pairs[i].L0;
    if (total > cap) return pd_fail(c, PD_ERR_CAPACITY, "pd_debug_candidates: more candidate lengths than `cap`");
    return 0;
}
