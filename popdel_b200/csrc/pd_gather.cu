// pd_gather.cu -- K2: active sets, per-sample upper-half medians and candidate deletion lengths of the flagged windows.
//
//   k_tile_q3      one warp = (flagged tile, sample), one LANE = one window of the tile: the read pairs that can be active
//                  in the tile are staged read group by read group in shared memory and scattered into per-window
//                  value lists; every lane then selects its window's Q3 (upperHalfMedian,
//                  genotype_deletion_popdel_call.h:15-27) by bisection on the value. Writes Q3, coverage state and the
//                  largest deviation per (window, sample) -- nothing else, so windows without candidates cost no pool.
//   k_tile_cmask   per flagged tile: the windows that got at least one candidate length, and their first row.
//   k_tile_gather  one warp = (tile with candidates, sample): active read pairs of the candidate windows -> pool
//                  (structure of arrays) + per read group offsets / counts, read by the EM kernels.
//   k_candidates   one block per flagged window: sort the Q3s over samples, gap-50 clustering with rank-indexed
//                  thresholds (:58-86) -> candidate initial lengths, kept inline per window.
//   k_cand_*       exclusive scan of the candidate counts -> (window, initial length) pairs in reference order.
#include "pd_device.cuh"

namespace {

constexpr int TG_WARPS = 4;
constexpr int TG_STAGE = 320;                                       // staged read pairs per warp
constexpr int TG_ACT = 96;                                          // active read pairs per (window, sample) via the fast path
constexpr int TG_MAXRG = 8;                                         // read groups per sample via the fast path

struct alignas(16) StagePair { int32_t s, e; uint32_t pos; int32_t dev; };

struct alignas(16) WarpStage {
    StagePair pair[TG_STAGE];
    uint16_t act[TG_ACT];
    uint32_t rg_first[TG_MAXRG + 1];
};

// upperHalfMedian (:15-27) from the order statistics l and l+1: n<4 -> the maximum; else interpolate at (3n+2+n%2)/4-1
__device__ __forceinline__ void q3_position(uint32_t nn, uint32_t & l, uint32_t & l2, double & r)
{
    r = 0;
    if (nn < 4) l = nn - 1;
    else { const double pos = (3.0 * nn + 2.0 + (nn % 2)) / 4.0 - 1.0; l = (uint32_t)pos; r = pos - l; }
    l2 = (l + 1 < nn) ? l + 1 : l;
}
__device__ __forceinline__ int32_t q3_value(uint32_t nn, double r, int32_t lo_v, int32_t hi_v)
{
    if (nn < 4) return (int32_t)floor((double)lo_v + 0.5);
    return (int32_t)floor((1 - r) * lo_v + r * hi_v + 0.5);
}

// ------------------------------------------------------------------------------------------------------------------
// K2a: Q3 of every (flagged window, sample)
// ------------------------------------------------------------------------------------------------------------------
constexpr int TQ_WARPS = 4;
// usable active read pairs per (window, sample) via the fast path: 48 (9 blocks per SM) for the passes over every flagged
// window; 92 for the pass over the few windows that survive the second screen stage -- they sit at deletions, where the
// carriers' spanning read pairs pile up and the slow path would dominate
template <int TQ_ACT>
struct alignas(16) WarpQ3 {
    int32_t val[32][TQ_ACT + 1];                                    // [window][slot]: deviations of the window's usable active pairs
    uint32_t cnt[32];                                               // (odd row stride: a lane per window and a lane per slot both hit 32 banks)
};
constexpr int TQ_COOP_MAX = 10;                                     // up to this many windows of a (tile, sample): one window at a time, whole warp

__device__ __forceinline__ void write_q3(const GatherArgs & ga, uint32_t N, uint32_t job, uint32_t smp, uint32_t cov, uint32_t n,
                                         int32_t q, int32_t mx)
{
    const size_t o = (size_t)job * N + smp;
    ga.q3[o] = (cov >= 2u && n) ? q : 0;
    ga.sstat[o] = cov < 2u ? 0 : (n == 0 ? 1 : 2);
    ga.dmax[o] = n ? mx : INT_MIN;
}

// Generic path of one (window, sample): no shared memory, any number of read pairs / read groups. The order
// statistics are found by bisection on the value, one pass over the read groups' tile batches per step.
__device__ __noinline__ void q3_window_slow(const PdDev & a, const GatherArgs & ga, uint32_t smp, int32_t w, uint32_t job, int lane)
{
    const uint32_t g0 = a.sample_rg[smp], g1 = a.sample_rg[smp + 1];
    const uint32_t tile = (uint32_t)w / PD_TILE_WINDOWS;
    // counts how many usable active deviations are <= t; also the smallest one above t
    auto pass = [&](int32_t t, uint32_t & cov, uint32_t & nvals, int32_t & mn, int32_t & mx, int32_t & above) {
        uint32_t c = 0;
        cov = 0; nvals = 0; mn = INT_MAX; mx = INT_MIN; above = INT_MAX;
        for (uint32_t g = g0; g < g1; ++g) {
            const PdRgConst k = a.rgc[g];
            uint32_t n_g = 0, c_g = 0; int32_t mn_g = INT_MAX, mx_g = INT_MIN, ab_g = INT_MAX;
            for_tile_batches(a, g, k, tile, lane, [&](bool valid, int32_t s, int32_t e, uint32_t, int32_t dev) {
                valid = valid && s <= w && w <= e;
                n_g += __popc(__ballot_sync(PD_FULL, valid));
                c_g += __popc(__ballot_sync(PD_FULL, valid && dev <= t));
                if (valid) { mn_g = min(mn_g, dev); mx_g = max(mx_g, dev); if (dev > t) ab_g = min(ab_g, dev); }
            });
            cov += n_g;
            if (n_g < k.max_load) { nvals += n_g; c += c_g; mn = min(mn, mn_g); mx = max(mx, mx_g); above = min(above, ab_g); }
        }
        for (int o = 16; o > 0; o >>= 1) {
            mn = min(mn, __shfl_xor_sync(PD_FULL, mn, o)); mx = max(mx, __shfl_xor_sync(PD_FULL, mx, o));
            above = min(above, __shfl_xor_sync(PD_FULL, above, o));
        }
        return c;
    };
    uint32_t cov, n; int32_t mn, mx, above;
    pass(INT_MAX, cov, n, mn, mx, above);
    int32_t q = 0;
    if (cov >= 2u && n) {
        uint32_t l, l2; double r;
        q3_position(n, l, l2, r);
        int32_t lo_v = mx, hi_v = mx;
        if (n >= 4) {
            int32_t lo = mn, hi = mx;
            uint32_t cov2, n2; int32_t a2, b2, ab2;
            while (lo < hi) {
                const int32_t mid = lo + (int32_t)(((uint32_t)hi - (uint32_t)lo) >> 1);
                if (pass(mid, cov2, n2, a2, b2, ab2) >= l + 1) hi = mid; else lo = mid + 1;
            }
            lo_v = lo;
            hi_v = pass(lo_v, cov2, n2, a2, b2, ab2) >= l2 + 1 ? lo_v : ab2;
        }
        q = q3_value(n, r, lo_v, hi_v);
    }
    if (lane == 0) write_q3(ga, a.N, job, smp, cov, n, q, mx);
}

// one (tile job, sample): Q3 of the windows of the tile this launch handles for the sample
template <int TQ_ACT>
__device__ __forceinline__ void q3_tile_job(const PdDev & a, const GatherArgs & ga, WarpQ3<TQ_ACT> & sh, int lane, uint32_t smp, uint32_t tjb)
{
    const uint32_t tj = ga.tj0 + tjb;
    const uint32_t tile = ga.tj_tile[tj], jmask = ga.tj_mask[tj];        // jmask numbers the window jobs of the tile
    // windows this launch handles for this sample (second screen stage: first the pairs whose Q3 can exceed t_known, later the
    // rest of the windows that survived)
    uint32_t wmask = jmask;
    if (ga.phase) {
        const uint32_t kn = ga.known[(size_t)smp * ga.known_stride + (tile - ga.tb_al)];
        wmask = ga.phase == 1 ? (jmask & kn) : (jmask & ga.tj_alive[tjb] & ~kn);
        if (wmask == 0) return;
        if (ga.phase == 1 && lane == 0) atomicAdd(&ga.counters[CNT_KNOWN], (uint32_t)__popc(wmask));
    }
    const uint32_t job_first = ga.tj_wbase[tj] - ga.job_base;            // scratch row of the tile's first flagged window
    const uint32_t g0 = a.sample_rg[smp], g1 = a.sample_rg[smp + 1];
    const int32_t w0 = (int32_t)(tile * PD_TILE_WINDOWS);
    const uint32_t lane_bit = 1u << lane;
    const uint32_t my_job = job_first + __popc(jmask & (lane_bit - 1u));

    sh.cnt[lane] = 0;
    uint32_t cov = 0;
    const bool slow = (ga.debug_flags & 1u) != 0;
    __syncwarp();
    for (uint32_t g = g0; g < g1 && !slow; ++g) {
        const PdRgConst k = a.rgc[g];
        const uint32_t before = sh.cnt[lane];
        __syncwarp();
        // every read pair appends its deviation to the lists of the flagged windows it is active in
        for_tile_batches(a, g, k, tile, lane, [&](bool valid, int32_t s, int32_t e, uint32_t, int32_t dev) {
            if (valid && e >= w0 && s <= w0 + 31) {
                const uint32_t sr = (uint32_t)max(s - w0, 0), er = (uint32_t)min(e - w0, 31);
                uint32_t m = wmask & (er == 31u ? 0xFFFFFFFFu : ((1u << (er + 1)) - 1u)) & ~((1u << sr) - 1u);
                while (m) {
                    const int w = __ffs(m) - 1;
                    m &= m - 1;
                    const uint32_t slot = atomicAdd(&sh.cnt[w], 1u);
                    if (slot < (uint32_t)TQ_ACT) sh.val[w][slot] = dev;
                }
            }
        });
        __syncwarp();
        const uint32_t n_g = sh.cnt[lane] - before;
        cov += n_g;
        if (n_g >= k.max_load) sh.cnt[lane] = before;                    // a high-coverage read group is left out (:1443-1478)
        __syncwarp();
    }
    const bool flagged = (wmask & lane_bit) != 0;
    const uint32_t n = sh.cnt[lane];
    const uint32_t over = __ballot_sync(PD_FULL, flagged && n > (uint32_t)TQ_ACT);
    uint32_t slow_mask = slow ? wmask : over;
    const uint32_t fast_mask = slow ? 0u : (wmask & ~over);
    if (__popc(fast_mask) <= TQ_COOP_MAX) {
        // Few windows (the second screen stage leaves 1-4 per tile): the warp takes them one at a time, a value (or two) per
        // lane, and pulls the largest values off with warp-wide max reductions until it holds the two order statistics --
        // Q3 sits in the top quarter, so that is n/4 + 1 reductions instead of a bisection that keeps one lane busy.
        for (uint32_t fm = fast_mask; fm; fm &= fm - 1) {
            const int w = __ffs(fm) - 1;
            const uint32_t nw = __shfl_sync(PD_FULL, n, w), cw = __shfl_sync(PD_FULL, cov, w);
            int32_t v0 = (uint32_t)lane < nw ? sh.val[w][lane] : INT_MIN, v1 = INT_MIN;
            if (nw > 32u && (uint32_t)lane + 32u < nw) v1 = sh.val[w][lane + 32];
            int32_t q = 0, mx = INT_MIN;
            if (nw) {
                uint32_t l, l2; double r;
                q3_position(nw, l, l2, r);
                const uint32_t t0 = nw - 1u - l, t1 = nw - 1u - l2;          // ranks from the top of v[l] >= ... and v[l2]
                int32_t lo_v = 0, hi_v = 0;
                const uint32_t steps = (cw >= 2u) ? t0 + 1u : 1u;
                for (uint32_t it = 0; it < steps; ++it) {
                    const int32_t cur = max(v0, v1);
                    const int32_t m = __reduce_max_sync(PD_FULL, cur);
                    if (it == 0) mx = m;
                    if (it == t1) hi_v = m;
                    if (it == t0) lo_v = m;
                    const uint32_t b = __ballot_sync(PD_FULL, cur == m);
                    if (lane == __ffs(b) - 1) { if (v0 == m) v0 = INT_MIN; else v1 = INT_MIN; }
                }
                if (cw >= 2u) q = q3_value(nw, r, lo_v, hi_v);
            }
            if (lane == w) write_q3(ga, a.N, my_job, smp, cov, n, q, mx);
        }
    } else if (flagged && n <= (uint32_t)TQ_ACT && !slow) {
        int32_t q = 0, mx = INT_MIN;
        if (cov >= 2u && n) {
            int32_t mn = INT_MAX;
            for (uint32_t i = 0; i < n; ++i) { const int32_t v = sh.val[lane][i]; mn = min(mn, v); mx = max(mx, v); }
            uint32_t l, l2; double r;
            q3_position(n, l, l2, r);
            int32_t lo_v = mx, hi_v = mx;
            if (n >= 4) {
                int32_t lo = mn, hi = mx;
                while (lo < hi) {                                        // smallest v with #{x <= v} >= l + 1
                    const int32_t mid = lo + (int32_t)(((uint32_t)hi - (uint32_t)lo) >> 1);
                    uint32_t c = 0;
                    for (uint32_t i = 0; i < n; ++i) c += sh.val[lane][i] <= mid;
                    if (c >= l + 1) hi = mid; else lo = mid + 1;
                }
                lo_v = lo;
                uint32_t c = 0; int32_t above = INT_MAX;
                for (uint32_t i = 0; i < n; ++i) { const int32_t v = sh.val[lane][i]; c += v <= lo_v; if (v > lo_v) above = min(above, v); }
                hi_v = c >= l2 + 1 ? lo_v : above;
            }
            q = q3_value(n, r, lo_v, hi_v);
        } else if (n) {
            for (uint32_t i = 0; i < n; ++i) mx = max(mx, sh.val[lane][i]);
        }
        write_q3(ga, a.N, my_job, smp, cov, n, q, mx);
    }
    __syncwarp();
    for (; slow_mask; slow_mask &= slow_mask - 1) {
        const int wl = __ffs(slow_mask) - 1;
        q3_window_slow(a, ga, smp, w0 + wl, job_first + __popc(jmask & ((1u << wl) - 1u)), lane);
    }
    __syncwarp();
}

template <int TQ_ACT, int MINB>
__global__ void __launch_bounds__(TQ_WARPS * 32, MINB) k_tile_q3(PdDev a, GatherArgs ga)
{
    __shared__ WarpQ3<TQ_ACT> sh_all[TQ_WARPS];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    if (ga.phase == 1 && ga.kjobs) {
        // second screen stage, first pass: the (sample, tile) pairs k_count listed, one per warp. (One warp per sample and a
        // loop over the tiles left three of a block's four warps idle wherever their samples' read groups sit far below the
        // threshold: 25 % active warps, ncu.)
        for (uint32_t i = (blockIdx.x + blockIdx.y * gridDim.x) * TQ_WARPS + wib; i < ga.n_kjobs; i += gridDim.x * gridDim.y * TQ_WARPS) {
            const uint2 e = ga.kjobs[i];
            const uint32_t tj = ga.tj_of_tile[e.y - ga.tile_begin];
            if (tj == 0xFFFFFFFFu || tj < ga.tj0 || tj >= ga.tj0 + ga.ntj) continue;      // no flagged window in the tile / another batch
            q3_tile_job<TQ_ACT>(a, ga, sh_all[wib], lane, e.x, tj - ga.tj0);
        }
        return;
    }
    const uint32_t smp = pd_grid_row() * TQ_WARPS + wib;
    if (smp >= a.N) return;
    // (blocks walk several tile jobs: with the second screen stage most (tile job, sample) pairs have nothing to do)
    for (uint32_t tjb = blockIdx.x; tjb < ga.ntj; tjb += gridDim.x) q3_tile_job<TQ_ACT>(a, ga, sh_all[wib], lane, smp, tjb);
}

// ------------------------------------------------------------------------------------------------------------------
// Second screen stage (cohorts with different thresholds per read group, where nearly every window has SOME sample whose
// Q3 can exceed the smallest one). initialize_deletion_lengths (:58-86) keeps a chain cluster only if its integer mean
// exceeds min T over its ranks >= t_min. Every Q3 that was NOT computed in phase 1 is <= t_known < t_min, so in the sorted
// array the values above t_known are exactly the phase-1 values above t_known, their chain clusters among themselves are
// exact, and the true cluster of a chain may only ADD values <= t_known below it, which lowers a mean that is above
// t_known. Hence: if no chain of the values above t_known has an integer mean above t_min, the window has no candidate.
// One warp per flagged window.
// ------------------------------------------------------------------------------------------------------------------
constexpr int S2_CAP = 256;                                         // values above t_known per window (more: the window survives)

__global__ void __launch_bounds__(256) k_screen2(PdDev a, GatherArgs ga)
{
    __shared__ int32_t s_val[8][S2_CAP], s_sorted[8][S2_CAP];
    __shared__ uint32_t s_alive;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t tj = ga.tj0 + blockIdx.x;
    const uint32_t tile = ga.tj_tile[tj], jmask = ga.tj_mask[tj];
    const uint32_t job_first = ga.tj_wbase[tj] - ga.job_base;
    if (threadIdx.x == 0) s_alive = 0;
    __syncthreads();
    uint32_t rank = 0;
    for (uint32_t m = jmask; m; m &= m - 1, ++rank) {
        if ((rank & 7u) != (uint32_t)wib) continue;
        const int wl = __ffs(m) - 1;
        const uint32_t job = job_first + rank;
        int32_t * val = s_val[wib], * srt = s_sorted[wib];
        uint32_t n = 0;
        for (uint32_t s0 = 0; s0 < a.N; s0 += 32) {
            const uint32_t s = s0 + lane;
            bool take = false; int32_t v = 0;
            if (s < a.N && ((ga.known[(size_t)s * ga.known_stride + (tile - ga.tb_al)] >> wl) & 1u)) {
                const size_t o = (size_t)job * a.N + s;
                if (ga.sstat[o] == 2) { v = ga.q3[o]; take = v > a.t_known; }
            }
            const uint32_t bm = __ballot_sync(PD_FULL, take);
            const uint32_t slot = n + __popc(bm & ((1u << lane) - 1u));
            if (take && slot < (uint32_t)S2_CAP) val[slot] = v;
            n += __popc(bm);
        }
        __syncwarp();
        bool alive = n > (uint32_t)S2_CAP;
        if (!alive && n) {
            for (uint32_t i = lane; i < n; i += 32) {                // rank sort (ties by index)
                const int32_t v = val[i];
                uint32_t r = 0;
                for (uint32_t j = 0; j < n; ++j) { const int32_t u = val[j]; r += (u < v) || (u == v && j < i); }
                srt[r] = v;
            }
            __syncwarp();
            if (lane == 0) {
                long long sum = srt[0]; int cnt = 1;
                for (uint32_t i = 1; i <= n; ++i) {
                    if (i < n && srt[i - 1] + 50 > srt[i]) { sum += srt[i]; ++cnt; continue; }
                    if ((int)(sum / cnt) > a.t_min) { alive = true; break; }
                    if (i < n) { sum = srt[i]; cnt = 1; }
                }
            }
            alive = __shfl_sync(PD_FULL, alive ? 1 : 0, 0) != 0;
        }
        if (lane == 0) {
            ga.job_dead[job] = alive ? 0 : 1;
            if (alive) atomicOr(&s_alive, 1u << wl);
        }
        __syncwarp();
    }
    __syncthreads();
    if (threadIdx.x == 0) { ga.tj_alive[blockIdx.x] = s_alive; if (s_alive) atomicAdd(&ga.counters[CNT_ALIVE], (uint32_t)__popc(s_alive)); }
}

// candidate windows of every flagged tile (after the candidate counts are known)
__global__ void __launch_bounds__(256) k_tile_cmask(GatherArgs ga, const uint32_t * __restrict__ cand_cnt, const uint32_t * __restrict__ cjob_of,
                                                    uint32_t * __restrict__ tj_cmask, uint32_t * __restrict__ tj_cfirst)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ga.ntj) return;
    const uint32_t tj = ga.tj0 + i;
    const uint32_t first = ga.tj_wbase[tj] - ga.job_base;
    uint32_t cm = 0, cf = 0xFFFFFFFFu, r = 0;
    for (uint32_t m = ga.tj_mask[tj]; m; m &= m - 1, ++r)
        if (cand_cnt[first + r]) { cm |= m & (0u - m); if (cf == 0xFFFFFFFFu) cf = cjob_of[first + r]; }
    tj_cmask[i] = cm; tj_cfirst[i] = cf;
}

// ------------------------------------------------------------------------------------------------------------------
// K2c: active sets of the candidate windows -> pool
// ------------------------------------------------------------------------------------------------------------------
// Generic (slow) path of one (window, sample): streams the read groups twice, no shared memory. Used when the staged
// list or the active set does not fit the fast path.
__device__ __noinline__ void gather_window_slow(const PdDev & a, const GatherArgs & ga, uint32_t smp, int32_t w, uint32_t row, int lane)
{
    const uint32_t g0 = a.sample_rg[smp], g1 = a.sample_rg[smp + 1];
    uint32_t * cnt = ga.act_cnt + (size_t)row * a.R;
    uint32_t * off = ga.act_off + (size_t)row * a.R;
    const uint32_t tile = (uint32_t)w / PD_TILE_WINDOWS;
    uint32_t nvals = 0;
    for (uint32_t g = g0; g < g1; ++g) {
        const PdRgConst k = a.rgc[g];
        uint32_t n_g = 0;
        for_tile_batches(a, g, k, tile, lane, [&](bool valid, int32_t s, int32_t e, uint32_t, int32_t) {
            n_g += __popc(__ballot_sync(PD_FULL, valid && s <= w && w <= e));
        });
        if (lane == 0) { cnt[g] = n_g; off[g] = nvals; }
        if (n_g < k.max_load) nvals += n_g;
    }
    uint32_t base = 0;
    if (lane == 0 && nvals) base = atomicAdd(&ga.counters[CNT_POOL], nvals);
    base = __shfl_sync(PD_FULL, base, 0);
    const bool fits = (uint64_t)base + nvals <= ga.pool_cap;
    __syncwarp();
    if (lane == 0) for (uint32_t g = g0; g < g1; ++g) off[g] += base;
    if (fits) {
        uint32_t cur = base;
        for (uint32_t g = g0; g < g1; ++g) {
            const PdRgConst k = a.rgc[g];
            const uint32_t n_g = __shfl_sync(PD_FULL, lane == 0 ? cnt[g] : 0u, 0);
            if (n_g >= k.max_load) continue;
            for_tile_batches(a, g, k, tile, lane, [&](bool valid, int32_t s, int32_t e, uint32_t pr, int32_t dev) {
                valid = valid && s <= w && w <= e;
                const uint32_t mask = __ballot_sync(PD_FULL, valid);
                if (valid) { const uint32_t i = cur + __popc(mask & ((1u << lane) - 1u)); ga.pool_pos[i] = pr; ga.pool_dev[i] = dev; }
                cur += __popc(mask);
            });
        }
    }
    __syncwarp();
}

__global__ void __launch_bounds__(TG_WARPS * 32) k_tile_gather(PdDev a, GatherArgs ga)
{
    __shared__ WarpStage stage_all[TG_WARPS];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t smp = pd_grid_row() * TG_WARPS + wib;
    if (smp >= a.N) return;
    const uint32_t wmask = ga.tj_cmask[blockIdx.x];                       // windows of the tile with candidate lengths
    const uint32_t cfirst = ga.tj_cfirst[blockIdx.x];
    if (wmask == 0 || cfirst < ga.cj_base || cfirst >= ga.cj_end) return;
    const uint32_t tile = ga.tj_tile[ga.tj0 + blockIdx.x];
    const uint32_t row_first = cfirst - ga.cj_base;                       // scratch row of the tile's first candidate window
    const uint32_t g0 = a.sample_rg[smp], g1 = a.sample_rg[smp + 1], nrg = g1 - g0;
    WarpStage & st = stage_all[wib];
    const int32_t w0 = (int32_t)(tile * PD_TILE_WINDOWS);

    // ---- stage every read pair whose interval intersects the tile (per read group, stream order)
    uint32_t total = 0;
    bool fast = nrg <= (uint32_t)TG_MAXRG && !(ga.debug_flags & 2u);
    if (fast) {
        for (uint32_t g = g0; g < g1; ++g) {
            if (lane == 0) st.rg_first[g - g0] = total;
            const PdRgConst k = a.rgc[g];
            for_tile_batches(a, g, k, tile, lane, [&](bool valid, int32_t s, int32_t e, uint32_t pr, int32_t dev) {
                valid = valid && e >= w0 && s <= w0 + 31;
                const uint32_t mask = __ballot_sync(PD_FULL, valid);
                const uint32_t slot = total + __popc(mask & ((1u << lane) - 1u));
                if (valid && slot < (uint32_t)TG_STAGE) st.pair[slot] = StagePair{s, e, pr, dev};
                total += __popc(mask);
            });
        }
        if (lane == 0) st.rg_first[nrg] = total;
        fast = total <= (uint32_t)TG_STAGE;
    }
    __syncwarp();

    // one pool reservation per (tile, sample): the staged read pairs' active windows among the candidate ones (an
    // upper bound of what is written: a high-coverage read group is left out of the pool)
    uint32_t tile_base = 0; bool tile_fits = true;
    if (fast) {
        uint32_t tot = 0;
        for (uint32_t i = lane; i < total; i += 32) {
            const int2 se = *reinterpret_cast<const int2 *>(&st.pair[i]);
            const int sr = max(se.x - w0, 0), er = min(se.y - w0, 31);
            tot += __popc(wmask & (er == 31 ? 0xFFFFFFFFu : ((1u << (er + 1)) - 1u)) & ~((1u << sr) - 1u));
        }
        for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(PD_FULL, tot, o);
        if (lane == 0 && tot) tile_base = atomicAdd(&ga.counters[CNT_POOL], tot);
        tile_base = __shfl_sync(PD_FULL, tile_base, 0);
        tile_fits = (uint64_t)tile_base + tot <= ga.pool_cap;
    }

    uint32_t rank = 0;
    for (uint32_t m = wmask; m; m &= m - 1, ++rank) {
        const int32_t w = w0 + (__ffs(m) - 1);
        const uint32_t row = row_first + rank;
        if (!fast) { gather_window_slow(a, ga, smp, w, row, lane); continue; }
        uint32_t * cnt = ga.act_cnt + (size_t)row * a.R;
        uint32_t * off = ga.act_off + (size_t)row * a.R;
        uint32_t nvals = 0;
        for (uint32_t gi = 0; gi < nrg; ++gi) {
            const uint32_t i_lo = st.rg_first[gi], i_hi = st.rg_first[gi + 1];
            uint32_t n_g = 0;
            for (uint32_t i0 = i_lo; i0 < i_hi; i0 += 32) {
                const uint32_t i = i0 + lane;
                bool valid = false;
                if (i < i_hi) { const int2 se = *reinterpret_cast<const int2 *>(&st.pair[i]); valid = se.x <= w && w <= se.y; }
                const uint32_t mask = __ballot_sync(PD_FULL, valid);
                const uint32_t slot = nvals + n_g + __popc(mask & ((1u << lane) - 1u));
                if (valid && slot < (uint32_t)TG_ACT) st.act[slot] = (uint16_t)i;
                n_g += __popc(mask);
            }
            if (lane == 0) { cnt[g0 + gi] = n_g; off[g0 + gi] = nvals; }
            if (n_g < __ldg(&a.rgc[g0 + gi].max_load)) nvals += n_g;          // a high-coverage read group is left out
        }
        if (nvals > (uint32_t)TG_ACT) { gather_window_slow(a, ga, smp, w, row, lane); continue; }
        const uint32_t base = tile_base;
        tile_base += nvals;
        __syncwarp();
        if ((uint32_t)lane < nrg) off[g0 + lane] += base;
        if (tile_fits)
            for (uint32_t i = lane; i < nvals; i += 32) {
                const StagePair p = st.pair[st.act[i]];
                ga.pool_pos[base + i] = p.pos; ga.pool_dev[base + i] = p.dev;
            }
        __syncwarp();                                                     // st.act is rewritten by the next window
    }
}

// ------------------------------------------------------------------------------------------------------------------
// K2b: candidates. One block per flagged window. mode 0: count + inline list; mode 1: windows with more than
// PD_CAND_INLINE candidates write their pairs directly (after the scan of the counts).
// ------------------------------------------------------------------------------------------------------------------
constexpr uint32_t CAND_BITS = 1u << 16;                     // value range the presence bitmap covers
constexpr uint32_t CAND_TOPS = 1024;                         // clusters per window via the bitmap path

struct CandEmit {
    const CandArgs & ca; uint32_t job; int mode; uint32_t pair0, nc;
    __device__ void operator()(int mean)
    {
        if (mode == 0) { if (nc < (uint32_t)PD_CAND_INLINE) ca.cand_inline[(size_t)job * PD_CAND_INLINE + nc] = mean; }
        else if (pair0 + nc < ca.pair_cap) ca.pairs[pair0 + nc] = PdPair{ca.job_base + job, mean};
        ++nc;
    }
};

// any value present in [lo, hi] (bit positions, hi - lo < 64)?
__device__ __forceinline__ bool bits_any(const uint32_t * bits, uint32_t lo, uint32_t hi)
{
    const uint32_t w0 = lo >> 5, w1 = hi >> 5;
    const uint32_t m0 = 0xFFFFFFFFu << (lo & 31u), m1 = 0xFFFFFFFFu >> (31u - (hi & 31u));
    if (w0 == w1) return (bits[w0] & m0 & m1) != 0;
    uint32_t r = (bits[w0] & m0) | (bits[w1] & m1);
    for (uint32_t w = w0 + 1; w < w1; ++w) r |= bits[w];
    return r != 0;
}

// f(Q3) of every sample of window `job` that has one (state 2), samples strided over the block's threads
template <typename F>
__device__ __forceinline__ void for_window_q3(const CandArgs & ca, uint32_t job, F f)
{
    for (uint32_t p = 0; p < ca.nparts; ++p) {
        const uint32_t np = ca.part_n[p];
        const uint8_t * ss = ca.sstat[p] + (size_t)job * np;
        const int32_t * qq = ca.q3[p] + (size_t)job * np;
        for (uint32_t s = threadIdx.x; s < np; s += blockDim.x)
            if (ss[s] == 2) f(qq[s]);
    }
}

// One block per flagged window: initialize_deletion_lengths (genotype_deletion_popdel_call.h:58-86) WITHOUT sorting the
// Q3 values. The chain clusters (sorted neighbours closer than 50) are the maximal runs of a presence bitmap over the
// value range whose gaps are shorter than 50: a value is the top of a cluster iff none of the next 49 values is
// present. Per cluster: sum and count by shared-memory atomics; the ranks of its members in the sorted array are
// [number of smaller values, + count), which is all the rank-indexed thresholds need (quirk, :65,72,80). Falls back to
// the bitonic sort for value ranges beyond 65 536 or more than 1 024 clusters.
// GLOBAL = false: the window's Q3s are copied once into dynamic shared memory (one int per sample of the cohort).
// GLOBAL = true (cohorts whose Q3s do not fit shared memory): every pass re-reads them from the Q3 / state rows in global
// memory; only the sorting fallback copies them, into this window's row of ca.sort_buf.
template <bool GLOBAL>
__global__ void __launch_bounds__(256) k_candidates(PdDev a, CandArgs ca, int mode)
{
    extern __shared__ int32_t s_q3[];
    __shared__ uint32_t s_bits[CAND_BITS / 32 + 4];
    __shared__ int32_t s_top[CAND_TOPS], s_sorted[CAND_TOPS], s_sum[CAND_TOPS];
    __shared__ uint32_t s_cnt[CAND_TOPS];
    __shared__ uint32_t s_n, s_ntop, s_thr, s_fill;
    __shared__ int32_t s_min, s_max;
    const uint32_t job = blockIdx.x;
    int32_t * const sv = GLOBAL ? ca.sort_buf + (size_t)job * ca.npad : s_q3;
    if (mode == 1 && ca.cand_cnt[job] <= (uint32_t)PD_CAND_INLINE) return;
    if (ca.job_dead && ca.job_dead[job]) { if (threadIdx.x == 0 && mode == 0) ca.cand_cnt[job] = 0; return; }      // rejected by the second screen stage
    if (threadIdx.x == 0) { s_n = 0; s_ntop = 0; s_min = INT_MAX; s_max = INT_MIN; if (GLOBAL) s_fill = 0; }
    __syncthreads();
    if (GLOBAL) {
        uint32_t n = 0; int32_t lo = INT_MAX, hi = INT_MIN;
        for_window_q3(ca, job, [&](int32_t v) { ++n; lo = min(lo, v); hi = max(hi, v); });
        if (n) { atomicAdd(&s_n, n); atomicMin(&s_min, lo); atomicMax(&s_max, hi); }
    } else {
        for_window_q3(ca, job, [&](int32_t v) { sv[atomicAdd(&s_n, 1u)] = v; atomicMin(&s_min, v); atomicMax(&s_max, v); });
    }
    __syncthreads();
    const uint32_t nv = s_n;
    if (nv == 0) { if (threadIdx.x == 0 && mode == 0) ca.cand_cnt[job] = 0; return; }
    // f(v) for every Q3 of the window, values strided over the block's threads
    auto each_value = [&](auto f) {
        if (GLOBAL) for_window_q3(ca, job, f);
        else for (uint32_t i = threadIdx.x; i < nv; i += blockDim.x) f(sv[i]);
    };
    CandEmit emit{ca, job, mode, mode == 1 ? ca.cand_off[job] : 0u, 0u};
    const int32_t mn = s_min;
    const uint32_t range = (uint32_t)(s_max - mn) + 1u;
    bool sorted_path = ca.force_sort || range > CAND_BITS;
    if (!sorted_path) {
        const uint32_t nwords = (range + 31) / 32;
        for (uint32_t w = threadIdx.x; w < nwords + 3; w += blockDim.x) s_bits[w] = 0;
        __syncthreads();
        each_value([&](int32_t v) { const uint32_t b = (uint32_t)(v - mn); atomicOr(&s_bits[b >> 5], 1u << (b & 31u)); });
        __syncthreads();
        for (uint32_t w = threadIdx.x; w < nwords; w += blockDim.x)
            for (uint32_t m = s_bits[w]; m; m &= m - 1) {
                const uint32_t b = w * 32 + (__ffs(m) - 1);
                if (!bits_any(s_bits, b + 1, b + 49)) { const uint32_t slot = atomicAdd(&s_ntop, 1u); if (slot < CAND_TOPS) s_top[slot] = (int32_t)b; }
            }
        __syncthreads();
        sorted_path = s_ntop > CAND_TOPS;
    }
    if (!sorted_path) {
        const uint32_t K = s_ntop;
        for (uint32_t t = threadIdx.x; t < K; t += blockDim.x) {
            const int32_t v = s_top[t];
            uint32_t r = 0;
            for (uint32_t u = 0; u < K; ++u) r += s_top[u] < v;
            s_sorted[r] = v; s_sum[t] = 0; s_cnt[t] = 0;
        }
        __syncthreads();
        each_value([&](int32_t v) {
            const int32_t b = v - mn;
            uint32_t lo = 0, hi = K - 1;                               // smallest k with top_k >= b
            while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (s_sorted[mid] >= b) hi = mid; else lo = mid + 1; }
            atomicAdd(&s_sum[lo], v); atomicAdd(&s_cnt[lo], 1u);
        });
        __syncthreads();
        uint32_t r0 = 0;
        for (uint32_t k = 0; k < K; ++k) {
            const uint32_t n = s_cnt[k];
            const int mean = s_sum[k] / (int)n;
            if (mean > a.t_min) {                                       // else it cannot exceed any threshold (t_min = their minimum)
                if (threadIdx.x == 0) s_thr = 0xFFFFFFFFu;
                __syncthreads();
                uint32_t t = 0xFFFFFFFFu;
                for (uint32_t i = r0 + threadIdx.x; i < r0 + n; i += blockDim.x) t = min(t, ca.min_init[i]);
                if (t != 0xFFFFFFFFu) atomicMin(&s_thr, t);
                __syncthreads();
                if (threadIdx.x == 0 && mean > (int)s_thr) emit(mean);
                __syncthreads();
            }
            r0 += n;
        }
        if (threadIdx.x == 0 && mode == 0) ca.cand_cnt[job] = emit.nc;
        return;
    }
    // ---- fallback: bitonic sort, then the reference's linear pass. Every compare-exchange sorts ascending (the first step
    // of a merge pairs i with its mirror image inside the block), so the padding up to the next power of two is virtual:
    // a partner at or beyond nv stands for +infinity and never moves -- sv holds nv values, not a power of two.
    if (GLOBAL) {                                                     // (in any order: the sort decides it)
        for_window_q3(ca, job, [&](int32_t v) { sv[atomicAdd(&s_fill, 1u)] = v; });
        __syncthreads();
    }
    uint32_t np2 = 1; while (np2 < nv) np2 <<= 1;
    for (uint32_t k = 2; k <= np2; k <<= 1)
        for (uint32_t j = k >> 1; j > 0; j >>= 1) {
            const uint32_t flip = (j == (k >> 1)) ? k - 1 : j;
            for (uint32_t i = threadIdx.x; i < nv; i += blockDim.x) {
                const uint32_t p = i ^ flip;
                if (p > i && p < nv) {
                    const int32_t x = sv[i], y = sv[p];
                    if (x > y) { sv[i] = y; sv[p] = x; }
                }
            }
            __syncthreads();
        }
    if (threadIdx.x == 0) {
        // genotype_deletion_popdel_call.h:62-84; thresholds are indexed by RANK in the sorted array (quirk)
        int sum = sv[0], n = 1;
        uint32_t thr = ca.min_init[0];
        for (uint32_t i = 1; i < nv; ++i) {
            if (sv[i - 1] + 50 > sv[i]) { sum += sv[i]; ++n; thr = min(thr, ca.min_init[i]); }
            else { if (sum / n > (int)thr) emit(sum / n); sum = sv[i]; n = 1; thr = ca.min_init[i]; }
        }
        if (sum / n > (int)thr) emit(sum / n);
        if (mode == 0) ca.cand_cnt[job] = emit.nc;
    }
}

// exclusive scan of cand_cnt -> cand_off, total -> counters[CNT_PAIRS]; inline candidates -> pairs. The same scan numbers
// the windows that have candidates (cjob_of, total -> counters[CNT_CJOBS]): value = pairs (low 40 bits) | windows << 40.
__device__ __forceinline__ unsigned long long cand_value(uint32_t c) { return c ? ((1ull << 40) | c) : 0ull; }
constexpr unsigned long long CAND_LOW = (1ull << 40) - 1;

__global__ void __launch_bounds__(1024) k_cand_sums(CandArgs ca)
{
    __shared__ unsigned long long ws[33];
    const uint32_t i = blockIdx.x * 1024 + threadIdx.x;
    unsigned long long total;
    block_excl_scan(cand_value(i < ca.njobs ? ca.cand_cnt[i] : 0u), ws, total);
    if (threadIdx.x == 0) ca.block_sums[blockIdx.x] = total;
}
__global__ void __launch_bounds__(1024) k_cand_offsets(CandArgs ca, uint32_t nb)
{
    __shared__ unsigned long long ws[33];
    unsigned long long carry = 0;
    for (uint32_t b0 = 0; b0 < nb; b0 += 1024) {
        const uint32_t b = b0 + threadIdx.x;
        unsigned long long total;
        const unsigned long long ex = block_excl_scan(b < nb ? ca.block_sums[b] : 0ull, ws, total);
        if (b < nb) ca.block_sums[b] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) {
        ca.counters[CNT_PAIRS] = (uint32_t)min(carry & CAND_LOW, 0xFFFFFFFFull);
        ca.counters[CNT_CJOBS] = (uint32_t)(carry >> 40);
    }
}
__global__ void __launch_bounds__(1024) k_cand_write(CandArgs ca)
{
    __shared__ unsigned long long ws[33];
    const uint32_t i = blockIdx.x * 1024 + threadIdx.x;
    const uint32_t c = i < ca.njobs ? ca.cand_cnt[i] : 0u;
    unsigned long long total;
    const unsigned long long ex = block_excl_scan(cand_value(c), ws, total) + ca.block_sums[blockIdx.x];
    if (i >= ca.njobs) return;
    const uint32_t o = (uint32_t)min(ex & CAND_LOW, 0xFFFFFFFFull);
    ca.cand_off[i] = o;
    ca.cjob_of[i] = (uint32_t)(ex >> 40);
    if (c <= (uint32_t)PD_CAND_INLINE)
        for (uint32_t k = 0; k < c; ++k)
            if (o + k < ca.pair_cap) ca.pairs[o + k] = PdPair{ca.job_base + i, ca.cand_inline[(size_t)i * PD_CAND_INLINE + k]};
}

}  // namespace

void pd_launch_q3(const PdDev & a, const GatherArgs & g, cudaStream_t st, uint64_t * launches)
{
    // (a 92-slot variant for the surviving windows of phase 2 was measured slower: 54.9 vs 49.9 ms per mixed 300 x 12 Mbp scan)
    const uint32_t gx = g.phase ? std::min<uint32_t>(g.ntj, 1024u) : g.ntj;
    if (g.phase == 1 && g.kjobs) {                                   // a list of (sample, tile) pairs: persistent-style grid
        const uint32_t nb = std::min<uint32_t>((g.n_kjobs + TQ_WARPS - 1) / TQ_WARPS, 148u * 9u * 8u);
        if (nb) k_tile_q3<48, 9><<<dim3(nb, 1), TQ_WARPS * 32, 0, st>>>(a, g);
        ++*launches;
        return;
    }
    k_tile_q3<48, 9><<<pd_rows_grid(gx, (a.N + TQ_WARPS - 1) / TQ_WARPS), TQ_WARPS * 32, 0, st>>>(a, g);
    ++*launches;
}

void pd_launch_screen2(const PdDev & a, const GatherArgs & g, cudaStream_t st, uint64_t * launches)
{
    k_screen2<<<g.ntj, 256, 0, st>>>(a, g);
    ++*launches;
}

void pd_launch_cmask(const GatherArgs & g, const CandArgs & ca, uint32_t * tj_cmask, uint32_t * tj_cfirst, cudaStream_t st, uint64_t * launches)
{
    k_tile_cmask<<<(g.ntj + 255) / 256, 256, 0, st>>>(g, ca.cand_cnt, ca.cjob_of, tj_cmask, tj_cfirst);
    ++*launches;
}

void pd_launch_gather(const PdDev & a, const GatherArgs & g, cudaStream_t st, uint64_t * launches)
{
    k_tile_gather<<<pd_rows_grid(g.ntj, (a.N + TG_WARPS - 1) / TG_WARPS), TG_WARPS * 32, 0, st>>>(a, g);
    ++*launches;
}

int pd_launch_candidates(pd_ctx * c, const PdDev & a, const CandArgs & ca, cudaStream_t st, uint64_t * launches)
{
    const bool global = ca.sort_buf != nullptr;
    if (!global && (size_t)ca.npad * 4 > 48 * 1024)
        PD_CUDA(c, cudaFuncSetAttribute(k_candidates<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(ca.npad * 4)));
    const uint32_t threads = ca.npad >= 512 ? 256 : (ca.npad >= 128 ? 64 : 32);
    const uint32_t nb = (ca.njobs + 1023) / 1024;
    if (global) k_candidates<true><<<ca.njobs, threads, 0, st>>>(a, ca, 0);
    else k_candidates<false><<<ca.njobs, threads, ca.npad * 4, st>>>(a, ca, 0);
    k_cand_sums<<<nb, 1024, 0, st>>>(ca);
    k_cand_offsets<<<1, 1024, 0, st>>>(ca, nb);
    k_cand_write<<<nb, 1024, 0, st>>>(ca);
    if (global) k_candidates<true><<<ca.njobs, threads, 0, st>>>(a, ca, 1);
    else k_candidates<false><<<ca.njobs, threads, ca.npad * 4, st>>>(a, ca, 1);
    *launches += 5;
    PD_CUDA(c, cudaGetLastError());
    return 0;
}
