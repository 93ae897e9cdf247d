// pd_screen.cu -- K1, the screen: which windows can have a candidate deletion length at all?
//
//   k_stream     (HBM-bound, the roofline kernel) reads every packed read-pair word of the window range exactly once
//                with 128-bit loads, one warp per granule of 1024 words, and only tests `dev > T_min` on the raw
//                word. A hit marks the (sample, tile) pairs whose windows the read pair can be active in (the tile is
//                found through the granule -> tile index; no per-tile table reads on the streaming path).
//   k_mark_long  marks the tiles reached by the wide-list read pairs (deletion-spanning pairs) above the threshold.
//   k_count      marked (sample, tile) pairs only: exact per-window counts of active read pairs (n) and of those above
//                the threshold (x), by a shared-memory difference histogram + warp scan; window passes iff cov >= 2, n >= 1 and x >= need(n) -- the exact necessary
//                condition for initialize_deletion_lengths (genotype_deletion_popdel_call.h:33-87) to return a
//                candidate (SURVEY.md App. E): some sample's upper-half median (:15-27) must exceed the smallest
//                initial-length threshold.
//   k_tj_*       ordered compaction of the flagged tiles into tile jobs / window jobs (two-level scan).
#include "pd_device.cuh"

namespace {

// ------------------------------------------------------------------------------------------------------------------
// granule index: gran_tile[gran_off[g] + j] = tile of read group g that contains word (first word of g) + j*PD_GRAN
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_gran_index(PdDev a, uint32_t * __restrict__ gran_tile, const uint32_t * __restrict__ gran_off)
{
    const uint64_t id = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= (uint64_t)a.NT * a.R) return;
    const uint32_t g = (uint32_t)(id / a.NT), t = (uint32_t)(id % a.NT);
    const PdTile * tl = a.tiles + (size_t)g * (a.NT + 1);
    const uint32_t base = tl[0].off, o0 = tl[t].off, o1 = tl[t + 1].off;
    if (o1 <= o0) return;
    uint32_t j = (o0 - base + PD_GRAN - 1) / PD_GRAN;
    uint32_t * out = gran_tile + gran_off[g];
    while ((uint64_t)base + (uint64_t)j * PD_GRAN < o1) { out[j] = t; ++j; }
}

__device__ __forceinline__ void mark_tiles(uint32_t * __restrict__ row, uint32_t lo, uint32_t hi, uint32_t tb_al)
{
    // sets the bits of tiles lo..hi (inclusive; at most 2 words apart for the look-back, any span for long read pairs)
    for (uint32_t w = (lo - tb_al) >> 5; w <= (hi - tb_al) >> 5; ++w) {
        const uint32_t first = max(lo - tb_al, w << 5) & 31u, last = min(hi - tb_al, (w << 5) + 31u) & 31u;
        const uint32_t mask = (last == 31u ? 0xFFFFFFFFu : ((1u << (last + 1)) - 1u)) & ~((1u << first) - 1u);
        if ((__ldcg(row + w) & mask) != mask) atomicOr(row + w, mask);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// K1a: stream. grid = (R, granule groups); one warp = one granule of PD_GRAN words = 8 x 128-bit loads per lane.
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_stream(PdDev a, ScreenArgs s)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t g = blockIdx.x;
    const PdTile * tl = a.tiles + (size_t)g * (a.NT + 1);
    const uint32_t lb = __ldg(&a.rgc[g].lookback_tiles);
    const uint32_t t_lo = s.tile_begin > lb ? s.tile_begin - lb : 0;
    const uint32_t base = __ldg(&tl[0].off), r0 = __ldg(&tl[t_lo].off), r1 = __ldg(&tl[s.tile_end].off);
    const uint32_t j = (r0 - base) / PD_GRAN + blockIdx.y * 8 + warp;
    const uint64_t a0l = (uint64_t)base + (uint64_t)j * PD_GRAN;
    if (a0l >= r1) return;
    const uint32_t a0 = (uint32_t)a0l, rem = r1 - a0;
    const int32_t thr = (int32_t)(((uint32_t)a.t_mark << 11) | 0x7FFu);     // (int)word > thr  <=>  dev > t_mark
    const uint4 * src = reinterpret_cast<const uint4 *>(a.words + a0) + lane;
    uint4 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        v[u] = make_uint4(PD_PAD_WORD, PD_PAD_WORD, PD_PAD_WORD, PD_PAD_WORD);
        if ((uint32_t)(u * 128 + lane * 4) < rem) v[u] = __ldcs(src + u * 32);          // streamed once: evict first
    }
    uint32_t ex = 0;
#pragma unroll
    for (int u = 0; u < 8; ++u)
        ex |= (uint32_t)(((int32_t)v[u].x > thr) | ((int32_t)v[u].y > thr) | ((int32_t)v[u].z > thr) | ((int32_t)v[u].w > thr)) << u;
    if (__ballot_sync(PD_FULL, ex != 0) == 0) return;

    // ---- rare path: find the tile of every 128-bit vector with a hit (tiles start at multiples of 4 words)
    const uint32_t th = __ldg(&s.gran_tile[__ldg(&s.gran_off[g]) + j]);
    const uint32_t te = th + lane;
    const uint32_t my_off = te <= a.NT ? __ldg(&tl[te].off) : 0xFFFFFFFFu;
    uint32_t * row = s.need + (size_t)__ldg(&a.rgc[g].sample) * s.need_stride;
    uint32_t last_tile = 0xFFFFFFFFu;
#pragma unroll 1
    for (int u = 0; u < 8; ++u) {
        uint32_t m = __ballot_sync(PD_FULL, (ex >> u) & 1u);
        while (m) {
            const int srcl = __ffs(m) - 1;
            m &= m - 1;
            const uint32_t wi = a0 + u * 128 + srcl * 4;
            const uint32_t cnt = __popc(__ballot_sync(PD_FULL, my_off <= wi));
            uint32_t tile = th + cnt - 1;
            if (cnt == 32 && th + 32 <= a.NT) {                      // beyond the staged entries: upper_bound(off, wi) - 1
                uint32_t lo = th + 32, hi = a.NT + 1;                // first entry with off > wi lies in [lo, hi]
                while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (__ldg(&tl[mid].off) <= wi) lo = mid + 1; else hi = mid; }
                tile = lo - 1;
            }
            if (tile == last_tile) continue;
            last_tile = tile;
            const uint32_t lo_t = max(tile, s.tile_begin), hi_t = min(tile + lb, s.tile_end - 1);
            if (lane == 0 && tile < s.tile_end && lo_t <= hi_t) mark_tiles(row, lo_t, hi_t, s.tb_al);
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// K1b: wide-list read pairs above the threshold mark every tile of their active interval. One thread per entry.
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_mark_long(PdDev a, ScreenArgs s)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= s.total_longs) return;
    const PdLong L = a.longs[i];
    if (L.dev <= a.t_mark) return;
    uint32_t lo = 0, hi = a.R;                                      // largest g with long_off[g] <= i
    while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (__ldg(&s.long_off[mid]) <= i) lo = mid; else hi = mid; }
    const uint32_t t0 = max(L.s / PD_TILE_WINDOWS, s.tile_begin), t1 = min(L.e / PD_TILE_WINDOWS, s.tile_end - 1);
    if (L.e / PD_TILE_WINDOWS < s.tile_begin || t0 > t1) return;
    mark_tiles(s.need + (size_t)a.rgc[lo].sample * s.need_stride, t0, t1, s.tb_al);
}

// ------------------------------------------------------------------------------------------------------------------
// K1c: exact counts of the marked (sample, tile) pairs. One warp = one word of the need bitmap (32 tiles of a sample).
// Per tile and read group the active intervals are clipped to the tile and histogrammed in shared memory (+1 at the
// first window, -1 after the last); an inclusive warp scan turns that into per-window counts (lane = window): n = active
// read pairs, x = those with dev > t_min.
// ------------------------------------------------------------------------------------------------------------------
struct CountHist { int n[33], x[33], y[33]; };        // y: read pairs above t_known (second stage)

__device__ __forceinline__ void count_tile(const PdDev & a, uint32_t g, const PdRgConst & k, uint32_t tile, int lane, CountHist & h,
                                           uint32_t & n_g, uint32_t & x_g, uint32_t & y_g)
{
    const int32_t w0 = (int32_t)(tile * PD_TILE_WINDOWS);
    const bool two = a.t_known != 0;
    h.n[lane] = 0; h.x[lane] = 0; h.y[lane] = 0;
    if (lane == 0) { h.n[32] = 0; h.x[32] = 0; h.y[32] = 0; }
    __syncwarp();
    for_tile_batches(a, g, k, tile, lane, [&](bool valid, int32_t s, int32_t e, uint32_t, int32_t dev) {
        if (valid && e >= w0 && s <= w0 + 31) {
            const int sr = max(s - w0, 0), er = min(e - w0, 31) + 1;
            atomicAdd(&h.n[sr], 1); atomicSub(&h.n[er], 1);
            if (dev > a.t_min) { atomicAdd(&h.x[sr], 1); atomicSub(&h.x[er], 1); }
            if (two && dev > a.t_known) { atomicAdd(&h.y[sr], 1); atomicSub(&h.y[er], 1); }
        }
    });
    __syncwarp();
    int n = h.n[lane], x = h.x[lane], y = h.y[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int pn = __shfl_up_sync(PD_FULL, n, o), px = __shfl_up_sync(PD_FULL, x, o), py = __shfl_up_sync(PD_FULL, y, o);
        if (lane >= o) { n += pn; x += px; y += py; }
    }
    n_g = (uint32_t)n; x_g = (uint32_t)x; y_g = (uint32_t)y;
    __syncwarp();
}

__global__ void __launch_bounds__(256) k_count(PdDev a, ScreenArgs s)
{
    __shared__ CountHist hist[8];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t wq = blockIdx.x * 8 + wib;
    if (wq >= s.need_stride) return;
    const uint32_t smp = pd_grid_row();                             // (samples over grid y and z: pd_rows_grid)
    if (smp >= a.N) return;
    uint32_t mq = s.need[(size_t)smp * s.need_stride + wq];
    if (mq == 0) return;
    const uint32_t g0 = a.sample_rg[smp], g1 = a.sample_rg[smp + 1];
    uint32_t kt = 0;                                                // tiles of this word with windows whose Q3 can exceed t_known
    while (mq) {
        const int b = __ffs(mq) - 1;
        mq &= mq - 1;
        const uint32_t tile = s.tb_al + wq * 32 + b;
        if (tile < s.tile_begin || tile >= s.tile_end) continue;
        uint32_t cov = 0, n = 0, x = 0, y = 0;
        for (uint32_t g = g0; g < g1; ++g) {
            const PdRgConst k = a.rgc[g];
            uint32_t n_g = 0, x_g = 0, y_g = 0;
            count_tile(a, g, k, tile, lane, hist[wib], n_g, x_g, y_g);
            cov += n_g;
            if (n_g < k.max_load) { n += n_g; x += x_g; y += y_g; }
        }
        const uint32_t w = tile * PD_TILE_WINDOWS + lane;
        const bool in = w >= a.w_begin && w < a.w_end && cov >= 2 && n >= 1;
        const bool pass = in && x >= pd_q3_need(n);
        const uint32_t pm = __ballot_sync(PD_FULL, pass);
        if (pm && lane == 0) atomicOr(&s.tile_flags[tile - s.tile_begin], pm);
        if (a.t_known != 0) {                                       // second stage: this sample's Q3 can exceed t_known in these windows
            const uint32_t km = __ballot_sync(PD_FULL, in && y >= pd_q3_need(n));
            if (lane == 0) s.known[(size_t)smp * (s.need_stride * 32) + (tile - s.tb_al)] = km;
            if (km) kt |= 1u << b;
        }
    }
    if (kt && s.kjobs) {                                            // one reservation per warp: the list phase 1 of k_tile_q3 walks
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(&s.counters[CNT_KJOBS], (uint32_t)__popc(kt));
        base = __shfl_sync(PD_FULL, base, 0);
        if ((kt >> lane) & 1u) {
            const uint32_t slot = base + __popc(kt & ((1u << lane) - 1u));
            if (slot < s.kjobs_cap) s.kjobs[slot] = make_uint2(smp, s.tb_al + wq * 32 + (uint32_t)lane);
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// pd_debug_device_window_sums: one warp per tile of read group g. Every read pair that for_tile_batches hands out and
// that is active in a window of [w_first, w_end) inside the tile adds its count, deviation and position to that window.
// ------------------------------------------------------------------------------------------------------------------
constexpr int WS_WARPS = 4;

__global__ void __launch_bounds__(WS_WARPS * 32) k_window_sums(PdDev a, uint32_t g, uint32_t anchor, uint32_t tile_begin, uint32_t tile_end,
                                                               uint64_t w_first, uint64_t w_end, unsigned long long * __restrict__ out)
{
    __shared__ unsigned long long sums[WS_WARPS][PD_TILE_WINDOWS * 3];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t tile = tile_begin + blockIdx.x * WS_WARPS + wib;
    if (tile >= tile_end) return;                                   // warp-uniform
    unsigned long long * sm = sums[wib];
    for (int i = lane; i < (int)PD_TILE_WINDOWS * 3; i += 32) sm[i] = 0;
    __syncwarp();
    const PdRgConst k = a.rgc[g];
    const int64_t w0 = (int64_t)tile * PD_TILE_WINDOWS;
    const int64_t lo = max(w0, (int64_t)w_first), hi = min(w0 + (int64_t)PD_TILE_WINDOWS - 1, (int64_t)w_end - 1);
    for_tile_batches(a, g, k, tile, lane, [&](bool valid, int32_t s, int32_t e, uint32_t pr, int32_t dev) {
        if (!valid) return;
        for (int64_t w = max((int64_t)s, lo); w <= min((int64_t)e, hi); ++w) {
            unsigned long long * o = sm + 3 * (w - w0);
            atomicAdd(o, 1ull);
            atomicAdd(o + 1, (unsigned long long)(long long)dev);
            atomicAdd(o + 2, (unsigned long long)pr + anchor);
        }
    });
    __syncwarp();
    for (int i = lane; i < (int)PD_TILE_WINDOWS * 3; i += 32) {
        const int64_t w = w0 + i / 3;
        if (w >= lo && w <= hi) out[3 * (w - (int64_t)w_first) + i % 3] = sm[i];
    }
}

// ------------------------------------------------------------------------------------------------------------------
// tile jobs: flagged tiles in ascending order with their window masks; window jobs numbered in ascending order
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long tj_value(const JobArgs & j, uint32_t t, uint32_t & mask)
{
    mask = t < j.n_tiles ? j.tile_flags[t] : 0u;
    return mask ? ((1ull << 32) | (unsigned long long)__popc(mask)) : 0ull;
}
__global__ void __launch_bounds__(1024) k_tj_sums(JobArgs j)
{
    __shared__ unsigned long long ws[33];
    uint32_t mask; unsigned long long total;
    block_excl_scan(tj_value(j, blockIdx.x * 1024 + threadIdx.x, mask), ws, total);
    if (threadIdx.x == 0) j.block_sums[blockIdx.x] = total;
}
__global__ void __launch_bounds__(1024) k_tj_offsets(JobArgs j, uint32_t nb)
{
    __shared__ unsigned long long ws[33];
    unsigned long long carry = 0;
    for (uint32_t b0 = 0; b0 < nb; b0 += 1024) {
        const uint32_t b = b0 + threadIdx.x;
        const unsigned long long v = b < nb ? j.block_sums[b] : 0ull;
        unsigned long long total;
        const unsigned long long ex = block_excl_scan(v, ws, total);
        if (b < nb) j.block_sums[b] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) { j.counters[CNT_TJOBS] = (uint32_t)(carry >> 32); j.counters[CNT_JOBS] = (uint32_t)carry; }
}
__global__ void __launch_bounds__(1024) k_tj_write(JobArgs j)
{
    __shared__ unsigned long long ws[33];
    const uint32_t t = blockIdx.x * 1024 + threadIdx.x;
    uint32_t mask; unsigned long long total;
    const unsigned long long ex = block_excl_scan(tj_value(j, t, mask), ws, total) + j.block_sums[blockIdx.x];
    if (!mask) return;
    const uint32_t k = (uint32_t)(ex >> 32), wb = (uint32_t)ex;
    j.tj_tile[k] = j.tile_begin + t; j.tj_mask[k] = mask; j.tj_wbase[k] = wb;
    if (j.tj_of_tile) j.tj_of_tile[t] = k;
    uint32_t r = 0;
    for (uint32_t m = mask; m; m &= m - 1, ++r) j.job_window[wb + r] = (j.tile_begin + t) * PD_TILE_WINDOWS + (__ffs(m) - 1);
}

}  // namespace

namespace {
__global__ void __launch_bounds__(256) k_tile_segs(uint4 * __restrict__ out, uint32_t n, uint32_t wb)
{
    const uint32_t t = blockIdx.x * 256 + threadIdx.x;
    if (t >= n) return;
    const TileSeg s = tile_seg(t, wb);
    out[t] = make_uint4(s.nb, (uint32_t)s.wlA, (uint32_t)s.wlB, (uint32_t)s.wlC);
}
}  // namespace

void pd_launch_tile_segs(uint4 * out, uint32_t n, uint32_t window_buffer, cudaStream_t st)
{
    k_tile_segs<<<(n + 255) / 256, 256, 0, st>>>(out, n, window_buffer);
}

void pd_launch_gran_index(const PdDev & a, uint32_t * gran_tile, const uint32_t * gran_off, cudaStream_t st)
{
    const uint64_t n = (uint64_t)a.NT * a.R;
    k_gran_index<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(a, gran_tile, gran_off);
}

void pd_launch_screen(const PdDev & a, const ScreenArgs & s, uint32_t max_rg_words, cudaStream_t st, cudaEvent_t after_stream, uint64_t * launches)
{
    const uint32_t granules = max_rg_words / PD_GRAN + 2;           // +1 partial granule, +1 for a range starting mid-granule
    k_stream<<<dim3(a.R, (granules + 7) / 8), 256, 0, st>>>(a, s);
    ++*launches;
    cudaEventRecord(after_stream, st);
    if (s.total_longs) { k_mark_long<<<(s.total_longs + 255) / 256, 256, 0, st>>>(a, s); ++*launches; }
    k_count<<<pd_rows_grid((s.need_stride + 7) / 8, a.N), 256, 0, st>>>(a, s);
    ++*launches;
}

void pd_launch_tile_jobs(const JobArgs & j, cudaStream_t st, uint64_t * launches)
{
    const uint32_t nb = (j.n_tiles + 1023) / 1024;
    k_tj_sums<<<nb, 1024, 0, st>>>(j);
    k_tj_offsets<<<1, 1024, 0, st>>>(j, nb);
    k_tj_write<<<nb, 1024, 0, st>>>(j);
    *launches += 3;
}

void pd_launch_window_sums(const PdDev & a, uint32_t g, uint32_t anchor, uint32_t tile_begin, uint32_t tile_end, uint64_t w_first,
                           uint64_t w_end, unsigned long long * out, cudaStream_t st)
{
    k_window_sums<<<(tile_end - tile_begin + WS_WARPS - 1) / WS_WARPS, WS_WARPS * 32, 0, st>>>(a, g, anchor, tile_begin, tile_end, w_first, w_end, out);
}
