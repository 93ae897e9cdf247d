// pd_pack.cu -- device-side packer: raw (pos, dev) arrays -> tiled 32-bit stream, tile table and wide list.
//
// Used by pd_contig_push_pinned(): the host only enqueues the H2D copies of the caller's page-locked arrays; tile
// boundaries (binary search), padded tile offsets (scan), the packed words, the wide list of long read pairs and its
// per-tile ranges are produced by the kernels below, with the same closed-form rule (pd_common.h) as the host packer.
// The active-coverage cap (ChromosomeProfile::add, profile_structure_popdel_call.h:1084-1113) is checked exactly on
// the device (open pairs at every read pair = i - #{lastWindow < bucket}); if it would drop anything, or a read pair
// spans more than the supported look-back, the contig is re-packed by the sequential host path instead.
#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

#include "pd_context.h"

#define PD_CUDA(c, call)                                                                          \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess)                                                                    \
            return pd_fail((c), PD_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

namespace {

constexpr int CAP_CHUNK_TILES = 32;
constexpr int CAP_MAX_LOOKBACK = 64;                       // tiles; beyond that the host path is used
constexpr int CAP_BINS = (CAP_MAX_LOOKBACK + CAP_CHUNK_TILES) * 32 + 32;

struct PackArgs {
    const uint32_t * pos; const int32_t * dev;             // raw arrays, all read groups
    const uint64_t * rg_start;                             // [R+1]
    const PdRgConst * rgc;
    uint32_t R, NT, anchor, window_buffer;
    uint32_t g0, ng;                                       // read groups handled by this launch
    uint32_t * tfirst;                                     // [R][NT+1] first read pair (RG-relative) of each tile
    uint32_t * flags;                                      // [0] unsorted, [1] cap would drop, [2] position before anchor
    uint32_t * span_tiles;                                 // [R] max (tile of last window - tile of the read pair)
};

// (all packing kernels work on the read groups [a.g0, a.g0 + a.ng) of one copy group)
__global__ void k_tile_first(PackArgs a)
{
    uint64_t id = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t per = (uint64_t)a.NT + 1;
    if (id >= per * a.ng) return;
    id += per * a.g0;
    const uint32_t g = (uint32_t)(id / per), t = (uint32_t)(id % per);
    const uint32_t * p = a.pos + a.rg_start[g];
    const uint64_t n = a.rg_start[g + 1] - a.rg_start[g];
    const uint64_t key = (uint64_t)a.anchor + (uint64_t)t * PD_TILE_BP;
    uint64_t lo = 0, hi = n;
    while (lo < hi) { const uint64_t mid = (lo + hi) >> 1; if ((uint64_t)p[mid] < key) lo = mid + 1; else hi = mid; }
    a.tfirst[id] = (uint32_t)lo;
}

// per read pair: order check and the largest tile span per read group. grid = (chunks of 1024 read pairs, read group)
__global__ void __launch_bounds__(256) k_check_span(PackArgs a)
{
    const uint32_t g = a.g0 + blockIdx.y;
    const uint64_t r0 = a.rg_start[g], n = a.rg_start[g + 1] - r0;
    const uint64_t first = (uint64_t)blockIdx.x * 1024;
    if (first >= n) return;
    const uint32_t * p = a.pos + r0;
    const int32_t * d = a.dev + r0;
    const int32_t inner_off = a.rgc[g].inner_off;
    const uint32_t lookback = a.rgc[g].lookback_tiles;
    uint32_t bad_order = 0, bad_anchor = 0, span_max = 0;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const uint64_t i = first + (uint64_t)u * 256 + threadIdx.x;
        if (i >= n) break;
        const uint32_t pi = __ldcs(p + i);
        if (pi < a.anchor) { bad_anchor = 1; continue; }
        if (i > 0 && __ldg(p + i - 1) > pi) bad_order = 1;
        const uint32_t pr = pi - a.anchor;
        int64_t inner = (int64_t)__ldcs(d + i) + inner_off;
        if (inner < 0) inner = 0;
        const uint64_t lw = ((uint64_t)pr + (uint64_t)inner) / PD_WIN;
        span_max = max(span_max, (uint32_t)min((uint64_t)0xFFFFu, (lw + 1) / PD_TILE_WINDOWS - pr / PD_TILE_BP));
    }
    if (bad_anchor) atomicOr(&a.flags[2], 1u);
    if (bad_order) atomicOr(&a.flags[0], 1u);
    if (span_max > lookback) atomicMax(&a.span_tiles[g], span_max);
}

// exact check of the active-coverage cap: one block per (read group, chunk of 32 tiles)
__global__ void __launch_bounds__(1024) k_cap_check(PackArgs a, uint32_t chunks_per_rg)
{
    __shared__ uint32_t hist[CAP_BINS + 1];
    __shared__ uint32_t wsum[32];
    const uint32_t g = a.g0 + blockIdx.x / chunks_per_rg, ch = blockIdx.x % chunks_per_rg;
    const uint32_t max_load = a.rgc[g].max_load;
    if (max_load == 0xFFFFFFFFu) return;
    const uint32_t kl = max(a.span_tiles[g], a.rgc[g].lookback_tiles);
    if (kl > CAP_MAX_LOOKBACK) return;                                    // host path decides (flagged by the caller)
    const uint32_t t0 = ch * CAP_CHUNK_TILES;
    if (t0 >= a.NT) return;
    const uint32_t t1 = min(t0 + CAP_CHUNK_TILES, a.NT);
    const uint32_t tl = t0 > kl ? t0 - kl : 0;
    const uint32_t * tf = a.tfirst + (size_t)g * (a.NT + 1);
    const uint32_t i_lo = tf[tl], i_mid = tf[t0], i_hi = tf[t1];
    if (i_hi - i_lo < max_load) return;                                   // cannot reach the cap at all
    const uint32_t * p = a.pos + a.rg_start[g];
    const int32_t * d = a.dev + a.rg_start[g];
    const int32_t inner_off = a.rgc[g].inner_off;
    const uint32_t w_lo = tl * PD_TILE_WINDOWS;
    const uint32_t nbins = (t1 - tl) * PD_TILE_WINDOWS + 1;              // last bin: last window beyond the chunk
    for (uint32_t b = threadIdx.x; b <= nbins; b += blockDim.x) hist[b] = 0;
    __syncthreads();
    for (uint32_t i = i_lo + threadIdx.x; i < i_hi; i += blockDim.x) {
        const uint32_t pr = p[i] - a.anchor;
        int64_t inner = (int64_t)d[i] + inner_off;
        if (inner < 0) inner = 0;
        const uint64_t lw = ((uint64_t)pr + (uint64_t)inner) / PD_WIN;
        const uint32_t bin = (uint32_t)min((uint64_t)(nbins - 1), lw - w_lo);
        atomicAdd(&hist[bin], 1u);
    }
    __syncthreads();
    // exclusive prefix sum over the bins: C[x] = number of read pairs in range with last window < w_lo + x
    uint32_t carry = 0;
    for (uint32_t base = 0; base < nbins; base += blockDim.x) {
        const uint32_t b = base + threadIdx.x;
        uint32_t v = b < nbins ? hist[b] : 0, inc = v;
        for (int o = 1; o < 32; o <<= 1) { uint32_t n = __shfl_up_sync(0xFFFFFFFFu, inc, o); if ((threadIdx.x & 31) >= o) inc += n; }
        if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = inc;
        __syncthreads();
        if (threadIdx.x < 32) {
            uint32_t s = wsum[threadIdx.x], si = s;
            for (int o = 1; o < 32; o <<= 1) { uint32_t n = __shfl_up_sync(0xFFFFFFFFu, si, o); if (threadIdx.x >= o) si += n; }
            wsum[threadIdx.x] = si - s;
        }
        __syncthreads();
        const uint32_t excl = carry + wsum[threadIdx.x >> 5] + inc - v;
        __syncthreads();
        if (b < nbins) hist[b] = excl;
        // total of this round
        if (threadIdx.x == blockDim.x - 1) wsum[0] = excl + v;
        __syncthreads();
        carry = wsum[0];
        __syncthreads();
    }
    bool bad = false;
    for (uint32_t i = i_mid + threadIdx.x; i < i_hi; i += blockDim.x) {
        const uint32_t b = (p[i] - a.anchor) / PD_WIN;
        const uint32_t open = (i - i_lo) - hist[b - w_lo];
        bad |= open >= max_load;
    }
    if (bad) atomicOr(&a.flags[1], 1u);
}

// padded tile sizes -> tile offsets (relative to the read group); one block per read group, sequential chunks
__global__ void __launch_bounds__(1024) k_tile_offsets(PackArgs a, uint32_t * rel_off /*[R][NT+1]*/, uint64_t * rg_words /*[R]*/)
{
    __shared__ uint32_t wsum[32];
    __shared__ uint32_t s_carry;
    const uint32_t g = a.g0 + blockIdx.x;
    const uint32_t * tf = a.tfirst + (size_t)g * (a.NT + 1);
    uint32_t * ro = rel_off + (size_t)g * (a.NT + 1);
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < a.NT; base += blockDim.x) {
        const uint32_t t = base + threadIdx.x;
        const uint32_t v = t < a.NT ? ((tf[t + 1] - tf[t] + 3u) & ~3u) : 0u;
        uint32_t inc = v;
        for (int o = 1; o < 32; o <<= 1) { uint32_t n = __shfl_up_sync(0xFFFFFFFFu, inc, o); if ((threadIdx.x & 31) >= o) inc += n; }
        if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = inc;
        __syncthreads();
        if (threadIdx.x < 32) {
            uint32_t s = wsum[threadIdx.x], si = s;
            for (int o = 1; o < 32; o <<= 1) { uint32_t n = __shfl_up_sync(0xFFFFFFFFu, si, o); if (threadIdx.x >= o) si += n; }
            wsum[threadIdx.x] = si - s;
        }
        __syncthreads();
        const uint32_t excl = s_carry + wsum[threadIdx.x >> 5] + inc - v;
        if (t < a.NT) ro[t] = excl;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) s_carry = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) { ro[a.NT] = s_carry; rg_words[g] = s_carry; }
}

struct WriteArgs {
    uint32_t * words; PdTile * tiles; PdLong * longs;
    const uint32_t * rel_off; const uint64_t * word_base;          // [R]
    uint32_t * lcount;                                              // [R][NT+1] long read pairs per tile -> offsets
    const uint64_t * long_base;                                     // [R]
    uint32_t * pmax;                                                // prefix max of e over the wide list
    uint32_t * reach;                                               // [R][NT+1] PdTile::reach (written by pass 0 of k_pack_tiles)
};

// one WARP per (read group, tile), lanes over the tile's read pairs (coalesced reads of the raw arrays, coalesced
// writes of the words): words, pads, count of long read pairs (pass 0) / wide entries in read order (pass 1)
__global__ void __launch_bounds__(256) k_pack_tiles(PackArgs a, WriteArgs w, int pass)
{
    uint64_t id = (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    const uint64_t per = (uint64_t)a.NT + 1;
    if (id >= per * a.ng) return;
    id += per * a.g0;
    const uint32_t g = (uint32_t)(id / per), t = (uint32_t)(id % per);
    if (t >= a.NT) { if (pass == 0 && lane == 0) { w.lcount[id] = 0; w.reach[id] = 0xFFFFFFu; } return; }
    if (pass == 1 && w.lcount[id + 1] == w.lcount[id]) return;            // no wide entries in this tile (the usual case)
    const PdRgConst k = a.rgc[g];
    const uint32_t * tf = a.tfirst + (size_t)g * per;
    const uint32_t * p = a.pos + a.rg_start[g];
    const int32_t * d = a.dev + a.rg_start[g];
    const uint32_t i0 = tf[t], i1 = tf[t + 1];
    uint32_t * out = w.words + w.word_base[g] + w.rel_off[id];
    PdLong * lout = pass == 1 ? w.longs + w.long_base[g] + w.lcount[id] : nullptr;
    uint32_t nl = 0, far = 0, first = 0xFFFFFFu;
    for (uint32_t base = i0; base < i1; base += 32) {
        const uint32_t i = base + lane;
        bool lng = false;
        uint32_t pr = 0; int32_t dv = 0; int64_t s = 0, e = 0;
        uint32_t ahead = 0;
        if (i < i1) {
            pr = __ldcs(p + i) - a.anchor;
            dv = __ldcs(d + i);
            const bool act = pd_interval(pr, dv, k.inner_off, a.window_buffer, s, e);
            bool is_long = dv > PD_DEV_MAX || dv < PD_DEV_MIN + 1;
            if (act && (uint64_t)e / PD_TILE_WINDOWS > (uint64_t)t + k.lookback_tiles) is_long = true;
            if (pass == 0) {
                const int32_t dc = dv > PD_DEV_MAX ? PD_DEV_MAX : (dv < PD_DEV_MIN + 1 ? PD_DEV_MIN + 1 : dv);
                out[i - i0] = pd_pack(dc, pr - t * PD_TILE_BP, is_long);
            }
            lng = is_long && act;
            if (act && !is_long && (uint64_t)e / PD_TILE_WINDOWS > t) ahead = (uint32_t)min((uint64_t)e / PD_TILE_WINDOWS - t, (uint64_t)255);
        }
        if (pass == 0) {
            const uint32_t rm = __ballot_sync(0xFFFFFFFFu, ahead != 0);
            if (rm && first == 0xFFFFFFu) first = min(base - i0 + (uint32_t)(__ffs(rm) - 1), 0xFFFFFFu);
            far = max(far, ahead);
        }
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, lng);
        if (pass == 1 && lng) lout[nl + __popc(m & ((1u << lane) - 1u))] = PdLong{(uint32_t)s, (uint32_t)e, pr, dv};
        nl += __popc(m);
    }
    if (pass == 0) {
        const uint32_t cnt = i1 - i0, padded = (cnt + 3u) & ~3u;
        if (cnt + lane < padded) out[cnt + lane] = PD_PAD_WORD;
        if (lane == 0) w.lcount[id] = nl;
        for (int o = 16; o > 0; o >>= 1) far = max(far, __shfl_xor_sync(0xFFFFFFFFu, far, o));
        if (lane == 0) w.reach[id] = (far << 24) | first;
    }
}

// wide entries in read order: one THREAD per (read group, tile) -- almost every tile has none and returns at once
__global__ void __launch_bounds__(256) k_pack_longs(PackArgs a, WriteArgs w)
{
    const uint64_t id = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t per = (uint64_t)a.NT + 1;
    if (id >= per * a.R) return;
    const uint32_t g = (uint32_t)(id / per), t = (uint32_t)(id % per);
    if (t >= a.NT || w.lcount[id + 1] == w.lcount[id]) return;
    const PdRgConst k = a.rgc[g];
    const uint32_t * tf = a.tfirst + (size_t)g * per;
    const uint32_t * p = a.pos + a.rg_start[g];
    const int32_t * d = a.dev + a.rg_start[g];
    PdLong * lout = w.longs + w.long_base[g] + w.lcount[id];
    uint32_t nl = 0;
    for (uint32_t i = tf[t]; i < tf[t + 1]; ++i) {
        const uint32_t pr = p[i] - a.anchor;
        const int32_t dv = d[i];
        int64_t s, e;
        const bool act = pd_interval(pr, dv, k.inner_off, a.window_buffer, s, e);
        bool is_long = dv > PD_DEV_MAX || dv < PD_DEV_MIN + 1;
        if (act && (uint64_t)e / PD_TILE_WINDOWS > (uint64_t)t + k.lookback_tiles) is_long = true;
        if (is_long && act) lout[nl++] = PdLong{(uint32_t)s, (uint32_t)e, pr, dv};
    }
}

// exclusive scan of lcount per read group (in place) and totals; one block per read group
__global__ void __launch_bounds__(1024) k_long_offsets(PackArgs a, uint32_t * lcount, uint64_t * rg_longs)
{
    __shared__ uint32_t wsum[32];
    __shared__ uint32_t s_carry;
    const uint32_t g = blockIdx.x;
    uint32_t * lc = lcount + (size_t)g * (a.NT + 1);
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base <= a.NT; base += blockDim.x) {
        const uint32_t t = base + threadIdx.x;
        const uint32_t v = t <= a.NT ? lc[t] : 0u;
        uint32_t inc = v;
        for (int o = 1; o < 32; o <<= 1) { uint32_t n = __shfl_up_sync(0xFFFFFFFFu, inc, o); if ((threadIdx.x & 31) >= o) inc += n; }
        if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = inc;
        __syncthreads();
        if (threadIdx.x < 32) {
            uint32_t s = wsum[threadIdx.x], si = s;
            for (int o = 1; o < 32; o <<= 1) { uint32_t n = __shfl_up_sync(0xFFFFFFFFu, si, o); if (threadIdx.x >= o) si += n; }
            wsum[threadIdx.x] = si - s;
        }
        __syncthreads();
        const uint32_t excl = s_carry + wsum[threadIdx.x >> 5] + inc - v;
        if (t <= a.NT) lc[t] = excl;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) s_carry = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) rg_longs[g] = s_carry;
}

// prefix maximum of e over each read group's wide list (lists are short: one thread per read group)
__global__ void k_long_pmax(PackArgs a, WriteArgs w, const uint64_t * rg_longs)
{
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= a.R) return;
    const PdLong * L = w.longs + w.long_base[g];
    uint32_t * pm = w.pmax + w.long_base[g];
    uint32_t m = 0;
    for (uint64_t i = 0; i < rg_longs[g]; ++i) { m = max(m, L[i].e); pm[i] = m; }
}

// tile table: word offset and the range [lo, hi) of wide entries that can be active in the tile
__global__ void k_tile_table(PackArgs a, WriteArgs w, const uint64_t * rg_longs)
{
    const uint64_t id = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t per = (uint64_t)a.NT + 1;
    if (id >= per * a.R) return;
    const uint32_t g = (uint32_t)(id / per), t = (uint32_t)(id % per);
    const PdLong * L = w.longs + w.long_base[g];
    const uint32_t * pm = w.pmax + w.long_base[g];
    const uint64_t n = rg_longs[g];
    const uint64_t w0 = (uint64_t)t * PD_TILE_WINDOWS;
    uint64_t lo = 0, hi = n;
    while (lo < hi) { const uint64_t mid = (lo + hi) >> 1; if ((uint64_t)L[mid].s <= w0 + PD_TILE_WINDOWS - 1) lo = mid + 1; else hi = mid; }
    const uint64_t hi_t = lo;
    lo = 0; hi = hi_t;
    while (lo < hi) { const uint64_t mid = (lo + hi) >> 1; if ((uint64_t)pm[mid] < w0) lo = mid + 1; else hi = mid; }
    PdTile tl;
    tl.off = (uint32_t)(w.word_base[g] + w.rel_off[id]);
    tl.long_lo = (uint32_t)(w.long_base[g] + lo);
    tl.long_hi = (uint32_t)(w.long_base[g] + hi_t);
    tl.reach = w.reach[id];
    w.tiles[id] = tl;
}

template <typename T>
int grow_dev(pd_ctx * c, int slot, T *& p, size_t need)
{
    size_t bytes = std::max<size_t>(need, 1) * sizeof(T);
    if (bytes > c->cap_pack[slot] || !c->d_pack[slot]) {
        if (c->d_pack[slot]) cudaFree(c->d_pack[slot]);
        c->d_pack[slot] = nullptr; c->cap_pack[slot] = 0;
        size_t want = bytes + bytes / 8 + 256;
        PD_CUDA(c, cudaMalloc(&c->d_pack[slot], want));
        c->cap_pack[slot] = want;
    }
    p = reinterpret_cast<T *>(c->d_pack[slot]);
    return 0;
}

}  // namespace

// Last window the reference scans (see last_scanned_window in pd_host.cu), from the tails of the raw host arrays.
// position / deviation of read pair i of a raw read group (either input form); `b` = block hint for compact input
static inline uint32_t raw_pos_at(const PdRawRg & r, uint64_t i, uint32_t & b)
{
    if (!r.compact()) return r.pos[i];
    if (r.w32 && (r.blk[b] > i || r.blk[b + 1] <= i)) {              // 256-bp blocks: search instead of walking
        uint32_t lo = 0, hi = r.nblk;
        while (hi - lo > 1) { const uint32_t m = lo + (hi - lo) / 2; if (r.blk[m] <= i) lo = m; else hi = m; }
        b = lo;
    }
    while (b > 0 && r.blk[b] > i) --b;
    while (b + 1 < r.nblk && r.blk[b + 1] <= i) ++b;
    return r.w32 ? ((b << 8) | (r.w32[i] & 0xFFu)) : ((b << 16) | r.lo[i]);
}
static inline int32_t raw_dev_at(const PdRawRg & r, uint64_t i)
{
    if (!r.compact()) return r.dev[i];
    if (r.w32) return (int32_t)r.w32[i] >> 8;
    const uint32_t u = (uint32_t)r.d24[3 * i] | ((uint32_t)r.d24[3 * i + 1] << 8) | ((uint32_t)r.d24[3 * i + 2] << 16);
    return (int32_t)(u << 8) >> 8;
}

// compact input (pd_contig_push_compact) -> the raw arrays the packing kernels read. grid (chunks of 4096 read pairs, read groups)
__global__ void __launch_bounds__(256) k_expand_compact(const uint16_t * __restrict__ lo, const uint8_t * __restrict__ d24, const uint32_t * __restrict__ blk,
                                                        const uint64_t * __restrict__ rg_start, const uint64_t * __restrict__ blk_start,
                                                        const uint32_t * __restrict__ rg_nblk, uint32_t g0, uint32_t * __restrict__ pos, int32_t * __restrict__ dev)
{
    const uint32_t g = g0 + blockIdx.y;
    const uint64_t s0 = rg_start[g], n = rg_start[g + 1] - s0;
    const uint64_t c0 = (uint64_t)blockIdx.x * 4096;
    if (c0 >= n) return;
    const uint32_t * bk = blk + blk_start[g];
    uint32_t nb = rg_nblk[g];
    const bool w32 = (nb >> 31) != 0;                              // 4-byte form: the words were copied into dev[], 256-bp blocks
    nb &= 0x7FFFFFFFu;
    if (nb == 0) return;                                           // this read group came as raw arrays
    for (uint64_t i = c0 + threadIdx.x; i < min(n, c0 + 4096); i += 256) {
        uint32_t a = 0, b = nb;                                   // largest block with blk[block] <= i
        while (b - a > 1) { const uint32_t m = (a + b) >> 1; if (__ldg(bk + m) <= i) a = m; else b = m; }
        if (w32) { const uint32_t w = (uint32_t)dev[s0 + i]; pos[s0 + i] = (a << 8) | (w & 0xFFu); dev[s0 + i] = (int32_t)w >> 8; continue; }
        pos[s0 + i] = (a << 16) | lo[s0 + i];
        const uint8_t * q = d24 + 3 * (s0 + i);
        const uint32_t u = (uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16);
        dev[s0 + i] = (int32_t)(u << 8) >> 8;
    }
}

// device-resident read groups (pd_contig_push_device): first / last position per read group, and the tail statistics
// last_window_from_raw takes from the host arrays
__global__ void __launch_bounds__(256) k_first_last(const uint32_t * const * __restrict__ pos, const uint64_t * __restrict__ n, uint32_t R, uint32_t * __restrict__ out)
{
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= R) return;
    out[2 * g] = 0; out[2 * g + 1] = 0;
    if (pos[g] && n[g]) { out[2 * g] = pos[g][0]; out[2 * g + 1] = pos[g][n[g] - 1]; }
}
// one block per read group: the read pairs of the last two segments (q >= start_km1) -> max S, E, E_spill (see last_window_from_raw)
__global__ void __launch_bounds__(256) k_tail_stats(const uint32_t * const * __restrict__ pos, const int32_t * const * __restrict__ dev, const uint64_t * __restrict__ n,
                                                    const PdRgConst * __restrict__ rgc, uint32_t anchor, long long start_kf, long long start_km1,
                                                    long long wl_kf, long long wl_km1, long long * __restrict__ out)
{
    const uint32_t g = blockIdx.x;
    const uint32_t * p = pos[g];
    if (!p || !n[g]) return;
    const int32_t * d = dev[g];
    const uint64_t cnt = n[g];
    uint64_t lo = 0, hi = cnt;                                       // first read pair with q >= start_km1 (positions are sorted)
    while (lo < hi) { const uint64_t mid = (lo + hi) >> 1; const uint32_t pr = p[mid] - anchor; if ((long long)(pr - pr % PD_WIN) < start_km1) lo = mid + 1; else hi = mid; }
    const int32_t io = rgc[g].inner_off;
    long long S = -1, E = -1, Esp = -1;
    for (uint64_t i = lo + threadIdx.x; i < cnt; i += blockDim.x) {
        const uint32_t pr = p[i] - anchor;
        const long long q = (long long)(pr - pr % PD_WIN);
        long long inner = (long long)d[i] + io; if (inner < 0) inner = 0;
        const long long lw = (long long)(((unsigned long long)pr + (unsigned long long)inner) / PD_WIN);
        if (q >= start_kf) { S = max(S, (long long)pr); if (lw <= wl_kf) E = max(E, lw); else Esp = max(Esp, lw); }
        else if (lw > wl_km1) E = max(E, lw);
    }
    if (S >= 0) atomicMax(&out[0], S);
    if (E >= 0) atomicMax(&out[1], E);
    if (Esp >= 0) atomicMax(&out[2], Esp);
}

static uint64_t last_window_from_raw(pd_ctx * c, const std::vector<uint32_t> & dev_first_last, int * rc)
{
    const uint32_t wb = c->grid.window_buffer, anchor = c->grid.anchor;
    c->tail = PdTail();
    int64_t kf = -1;
    bool any_dev = false;
    for (uint32_t g = 0; g < c->R; ++g) {
        const PdRawRg & r = c->raw[g];
        uint32_t bh = r.nblk ? r.nblk - 1 : 0;
        if (!r.n) continue;
        any_dev = any_dev || r.on_device;
        const uint32_t last = r.on_device ? dev_first_last[2 * g + 1] : raw_pos_at(r, r.n - 1, bh);
        kf = std::max<int64_t>(kf, (int64_t)((uint64_t)((last - anchor) / PD_WIN) * PD_WIN / wb));
    }
    if (kf < 0) return 0;
    int64_t E = -1, S = -1, Esp = -1;
    // segment of a read pair = floor(30 * floor(pr / 30) / wb): compare 30 * floor(pr / 30) with the segment starts
    // instead of dividing per read pair (this loop walks the last two segments of every read group on the host)
    const int64_t start_kf = kf * (int64_t)wb, start_km1 = (kf - 1) * (int64_t)wb;
    const int64_t wl_kf = (int64_t)pd_seg_last_window((uint64_t)kf, wb), wl_km1 = kf > 0 ? (int64_t)pd_seg_last_window((uint64_t)(kf - 1), wb) : -1;
    if (any_dev) {                                                  // device-resident read groups: reduced on the device
        long long * d_out = reinterpret_cast<long long *>(c->d_pack[12]) + 0;
        const uint32_t * const * d_ptrs = reinterpret_cast<const uint32_t * const *>(reinterpret_cast<char *>(c->d_pack[12]) + 64);
        const int32_t * const * d_dptrs = reinterpret_cast<const int32_t * const *>(d_ptrs + c->R);
        const uint64_t * d_n = reinterpret_cast<const uint64_t *>(d_dptrs + c->R);
        long long init[3] = {-1, -1, -1}, got[3];
        cudaError_t e = cudaMemcpyAsync(d_out, init, sizeof(init), cudaMemcpyHostToDevice, c->stream);
        k_tail_stats<<<c->R, 256, 0, c->stream>>>(d_ptrs, d_dptrs, d_n, c->d_rgc, anchor, start_kf, start_km1, wl_kf, wl_km1, d_out);
        if (e == cudaSuccess) e = cudaMemcpyAsync(got, d_out, sizeof(got), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) { *rc = pd_fail(c, PD_ERR_CUDA, std::string("pd_contig_push_device: ") + cudaGetErrorString(e)); return 0; }
        S = got[0]; E = got[1]; Esp = got[2];
    }
    for (uint32_t g = 0; g < c->R; ++g) {
        const PdRawRg & r = c->raw[g];
        if (r.on_device) continue;
        const int32_t io = c->rgc[g].inner_off;
        uint32_t bh = r.nblk ? r.nblk - 1 : 0;
        for (uint64_t i = r.n; i-- > 0;) {
            const uint32_t pr = raw_pos_at(r, i, bh) - anchor;
            const int64_t q = (int64_t)(pr - pr % PD_WIN);
            if (q < start_km1) break;
            const int64_t inner = std::max<int64_t>(0, (int64_t)raw_dev_at(r, i) + io);
            const int64_t lw = (int64_t)(((uint64_t)pr + (uint64_t)inner) / PD_WIN);
            if (q >= start_kf) { S = std::max<int64_t>(S, (int64_t)pr); if (lw <= wl_kf) E = std::max(E, lw); else Esp = std::max(Esp, lw); }
            else if (lw > wl_km1) E = std::max(E, lw);
        }
    }
    c->tail.kf = kf; c->tail.S = S; c->tail.E = E; c->tail.E_spill = Esp;
    return pd_tail_windows(c->tail, wb);
}

// returns 0 on success, 1 when the contig must be packed by the host path instead, <0 on error
int pd_pack_on_device(pd_ctx * c)
{
    PD_CUDA(c, cudaSetDevice(c->device));
    const uint32_t R = c->R;
    std::vector<uint64_t> rg_start(R + 1, 0);
    uint32_t max_pos_rel = 0; bool any = false, any_compact = false, any_device = false;
    for (uint32_t g = 0; g < R; ++g) any_device = any_device || (c->raw[g].on_device && c->raw[g].n);
    std::vector<uint32_t> dev_fl;
    if (any_device) {                                               // slot 12: tail statistics | pos pointers | dev pointers | counts | first/last
        char * d_meta = nullptr;
        if (grow_dev(c, 12, d_meta, 64 + (size_t)R * 32)) return c->status;
        std::vector<const uint32_t *> hp(R, nullptr); std::vector<const int32_t *> hd(R, nullptr); std::vector<uint64_t> hn(R, 0);
        for (uint32_t g = 0; g < R; ++g) if (c->raw[g].on_device) { hp[g] = c->raw[g].pos; hd[g] = c->raw[g].dev; hn[g] = c->raw[g].n; }
        PD_CUDA(c, cudaMemcpyAsync(d_meta + 64, hp.data(), (size_t)R * 8, cudaMemcpyHostToDevice, c->stream));
        PD_CUDA(c, cudaMemcpyAsync(d_meta + 64 + (size_t)R * 8, hd.data(), (size_t)R * 8, cudaMemcpyHostToDevice, c->stream));
        PD_CUDA(c, cudaMemcpyAsync(d_meta + 64 + (size_t)R * 16, hn.data(), (size_t)R * 8, cudaMemcpyHostToDevice, c->stream));
        uint32_t * d_fl = reinterpret_cast<uint32_t *>(d_meta + 64 + (size_t)R * 24);
        k_first_last<<<(R + 255) / 256, 256, 0, c->stream>>>(reinterpret_cast<const uint32_t * const *>(d_meta + 64),
                                                             reinterpret_cast<const uint64_t *>(d_meta + 64 + (size_t)R * 16), R, d_fl);
        dev_fl.resize((size_t)2 * R);
        PD_CUDA(c, cudaMemcpyAsync(dev_fl.data(), d_fl, (size_t)R * 8, cudaMemcpyDeviceToHost, c->stream));
        PD_CUDA(c, cudaStreamSynchronize(c->stream));               // (hp / hd / hn are host vectors read by the async copies)
    }
    for (uint32_t g = 0; g < R; ++g) {
        const PdRawRg & r = c->raw[g];
        rg_start[g + 1] = rg_start[g] + r.n;
        if (r.n) {
            uint32_t b0 = 0, b1 = r.nblk ? r.nblk - 1 : 0;
            const uint32_t first = r.on_device ? dev_fl[2 * g] : raw_pos_at(r, 0, b0), last = r.on_device ? dev_fl[2 * g + 1] : raw_pos_at(r, r.n - 1, b1);
            if (first < c->grid.anchor) return pd_fail(c, PD_ERR_ARG, "pd_contig_push_pinned: position before the contig anchor");
            if (last < c->grid.anchor) return pd_fail(c, PD_ERR_ARG, "pd_contig_push_device: position before the contig anchor");
            max_pos_rel = std::max(max_pos_rel, last - c->grid.anchor); any = true;
        }
        any_compact = any_compact || r.compact();
    }
    const uint64_t total = rg_start[R];
    if (total > 0xFFFFFFF0ull) return pd_fail(c, PD_ERR_CAPACITY, "more than 2^32 read pairs in one contig batch");
    cudaStream_t st = c->stream;
    uint32_t * d_pos = nullptr; int32_t * d_dev = nullptr; uint64_t * d_u64 = nullptr; uint32_t * d_tfirst = nullptr, * d_rel = nullptr, * d_lcount = nullptr, * d_small = nullptr, * d_pmax = nullptr;
    if (grow_dev(c, 0, d_pos, total)) return c->status;
    if (grow_dev(c, 1, d_dev, total)) return c->status;
    // compact input: staging of the 16-bit remainders, 24-bit deviations and block tables
    uint16_t * d_lo = nullptr; uint8_t * d_d24 = nullptr; uint32_t * d_blk = nullptr, * d_nblk = nullptr; uint64_t * d_blk_start = nullptr;
    std::vector<uint64_t> blk_start(R + 1, 0);
    std::vector<uint32_t> h_nblk(R, 0);
    if (any_compact) {
        for (uint32_t g = 0; g < R; ++g) {
            const uint32_t nb = c->raw[g].compact() ? c->raw[g].nblk : 0;
            h_nblk[g] = nb | (nb && c->raw[g].w32 ? 0x80000000u : 0u);
            blk_start[g + 1] = blk_start[g] + (nb ? nb + 1 : 0);
        }
        bool any5 = false;                                         // the 5-byte form needs its own staging, the 4-byte form lands in dev[]
        for (uint32_t g = 0; g < R; ++g) any5 = any5 || (c->raw[g].lo != nullptr && c->raw[g].n);
        if (grow_dev(c, 8, d_lo, any5 ? total : 1) || grow_dev(c, 9, d_d24, any5 ? total * 3 + 4 : 4) || grow_dev(c, 10, d_blk, blk_start[R] + 1) ||
            grow_dev(c, 11, d_blk_start, (size_t)2 * (R + 1))) return c->status;
        d_nblk = reinterpret_cast<uint32_t *>(d_blk_start + (R + 1));
    }

    // ---- copy groups of about equal read-pair counts: all copies are queued on the copy stream FIRST; the host-side
    // preparation below and the packing kernels of group k then overlap the PCIe transfer of the later groups
    constexpr int PACK_GROUPS = 8;
    if (!c->ev_pack[0]) for (auto & e : c->ev_pack) PD_CUDA(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    cudaStream_t cp = c->stream2;
    PD_CUDA(c, cudaEventRecord(c->ev[0], st));
    PD_CUDA(c, cudaEventRecord(c->ev_pack[PACK_GROUPS], st));             // the copy stream starts after everything queued before
    PD_CUDA(c, cudaStreamWaitEvent(cp, c->ev_pack[PACK_GROUPS], 0));
    uint32_t grp_lo[PACK_GROUPS + 1]; uint64_t grp_max[PACK_GROUPS];
    uint64_t h2d = 0;
    int n_groups = 0;
    for (uint32_t g_lo = 0; n_groups < PACK_GROUPS && g_lo < R; ++n_groups) {
        const int k = n_groups;
        const uint64_t target = rg_start[g_lo] + (total - rg_start[g_lo] + (PACK_GROUPS - k) - 1) / (PACK_GROUPS - k);
        uint32_t g_hi = g_lo + 1;
        while (g_hi < R && (k == PACK_GROUPS - 1 || rg_start[g_hi + 1] <= target)) ++g_hi;
        grp_lo[k] = g_lo; grp_max[k] = 0;
        for (uint32_t g = g_lo; g < g_hi; ++g) {
            const PdRawRg & r = c->raw[g];
            grp_max[k] = std::max<uint64_t>(grp_max[k], r.n);
            if (!r.n) continue;
            if (r.w32) {                                           // the words go straight into dev[]; k_expand_compact splits them in place
                PD_CUDA(c, cudaMemcpyAsync(d_dev + rg_start[g], r.w32, r.n * 4, cudaMemcpyHostToDevice, cp));
                PD_CUDA(c, cudaMemcpyAsync(d_blk + blk_start[g], r.blk, ((size_t)r.nblk + 1) * 4, cudaMemcpyHostToDevice, cp));
                h2d += r.n * 4 + ((size_t)r.nblk + 1) * 4;
                continue;
            }
            if (r.compact()) {
                PD_CUDA(c, cudaMemcpyAsync(d_lo + rg_start[g], r.lo, r.n * 2, cudaMemcpyHostToDevice, cp));
                PD_CUDA(c, cudaMemcpyAsync(d_d24 + 3 * rg_start[g], r.d24, r.n * 3, cudaMemcpyHostToDevice, cp));
                PD_CUDA(c, cudaMemcpyAsync(d_blk + blk_start[g], r.blk, ((size_t)r.nblk + 1) * 4, cudaMemcpyHostToDevice, cp));
                h2d += r.n * 5 + ((size_t)r.nblk + 1) * 4;
                continue;
            }
            if (!r.on_device) h2d += r.n * 8;
            const cudaMemcpyKind kind = r.on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
            PD_CUDA(c, cudaMemcpyAsync(d_pos + rg_start[g], r.pos, r.n * 4, kind, cp));
            PD_CUDA(c, cudaMemcpyAsync(d_dev + rg_start[g], r.dev, r.n * 4, kind, cp));
        }
        PD_CUDA(c, cudaEventRecord(c->ev_pack[k], cp));
        g_lo = g_hi;
        grp_lo[k + 1] = g_hi;
    }

    int tail_rc = 0;
    c->n_windows_total = any ? last_window_from_raw(c, dev_fl, &tail_rc) : 0;
    if (tail_rc) return tail_rc;
    const uint32_t NT = (uint32_t)std::max<uint64_t>(std::max<uint64_t>((std::max(c->n_windows_total, c->min_windows) + PD_TILE_WINDOWS - 1) / PD_TILE_WINDOWS,
                                                                        any ? (uint64_t)max_pos_rel / PD_TILE_BP + 1 : 0), 1);
    c->NT = NT;
    const size_t per = (size_t)NT + 1;
    if (grow_dev(c, 2, d_u64, (size_t)5 * (R + 1))) return c->status;        // rg_start | rg_words | word_base | rg_longs | long_base
    if (grow_dev(c, 3, d_tfirst, per * R)) return c->status;
    if (grow_dev(c, 4, d_rel, per * R)) return c->status;
    if (grow_dev(c, 5, d_lcount, per * R)) return c->status;
    if (grow_dev(c, 6, d_small, (size_t)R + 16)) return c->status;           // flags[4] | span_tiles[R]
    uint64_t * d_rg_start = d_u64, * d_rg_words = d_u64 + (R + 1), * d_word_base = d_u64 + 2 * (R + 1),
             * d_rg_longs = d_u64 + 3 * (R + 1), * d_long_base = d_u64 + 4 * (R + 1);
    // ---- word bases from UPPER BOUNDS of the packed sizes (every non-empty tile pads to a multiple of 4 words), so that
    // packing needs no host round trip and can start while later read groups are still crossing PCIe
    const uint64_t ntile = per * R;
    std::vector<uint64_t> base(R + 1, 0);
    uint64_t max_n = 0;
    for (uint32_t g = 0; g < R; ++g) {
        const uint64_t n = c->raw[g].n;
        base[g + 1] = base[g] + ((n + 3 * std::min<uint64_t>(NT, n) + 3) & ~3ull);
        max_n = std::max(max_n, n);
    }
    if (base[R] > 0xFFFFFFF0ull) return pd_fail(c, PD_ERR_CAPACITY, "more than 2^32 packed words in one contig batch; split the cohort or the contig");
    c->total_words = base[R];
    c->h_word_base = base;
    c->n_reads = total;
    if (c->total_words + 4 > c->cap_words || !c->d_words) {
        if (c->d_words) cudaFree(c->d_words);
        c->d_words = nullptr; c->cap_words = 0;
        size_t want = c->total_words + c->total_words / 8 + 1024;
        PD_CUDA(c, cudaMalloc(&c->d_words, want * 4));
        c->cap_words = want;
    }
    PD_CUDA(c, cudaMemcpyAsync(d_rg_start, rg_start.data(), (R + 1) * 8, cudaMemcpyHostToDevice, st));
    PD_CUDA(c, cudaMemcpyAsync(d_word_base, base.data(), (R + 1) * 8, cudaMemcpyHostToDevice, st));
    PD_CUDA(c, cudaMemsetAsync(d_small, 0, ((size_t)R + 16) * 4, st));
    c->h2d_bytes = h2d + (R + 1) * 16;
    if (any_compact) {
        PD_CUDA(c, cudaMemcpyAsync(d_blk_start, blk_start.data(), (R + 1) * 8, cudaMemcpyHostToDevice, st));
        PD_CUDA(c, cudaMemcpyAsync(d_nblk, h_nblk.data(), (size_t)R * 4, cudaMemcpyHostToDevice, st));
    }

    PackArgs a;
    a.pos = d_pos; a.dev = d_dev; a.rg_start = d_rg_start; a.rgc = c->d_rgc; a.R = R; a.NT = NT; a.g0 = 0; a.ng = R;
    a.anchor = c->grid.anchor; a.window_buffer = c->grid.window_buffer; a.tfirst = d_tfirst; a.flags = d_small; a.span_tiles = d_small + 16;
    WriteArgs w;
    w.words = c->d_words; w.tiles = nullptr; w.longs = nullptr; w.rel_off = d_rel; w.word_base = d_word_base;
    w.lcount = d_lcount; w.long_base = d_long_base; w.pmax = nullptr;
    if (grow_dev(c, 13, w.reach, per * R)) return c->status;
    const uint32_t chunks = (NT + CAP_CHUNK_TILES - 1) / CAP_CHUNK_TILES;

    // ---- per copy group, as soon as its raw arrays have arrived: order / span check, tile search, coverage-cap check,
    // tile offsets, words
    for (int k = 0; k < n_groups; ++k) {
        PD_CUDA(c, cudaStreamWaitEvent(st, c->ev_pack[k], 0));
        a.g0 = grp_lo[k]; a.ng = grp_lo[k + 1] - grp_lo[k];
        const uint64_t nt_grp = per * a.ng;
        for (uint32_t g = 0; g < a.ng; g += 65535) {                     // (gridDim.y: at most 65 535 read groups per launch)
            PackArgs b = a;
            b.g0 = a.g0 + g; b.ng = std::min<uint32_t>(a.ng - g, 65535);
            if (any_compact && grp_max[k])       // (read groups pushed as raw arrays have no blocks: their chunks exit at once)
                k_expand_compact<<<dim3((unsigned)((grp_max[k] + 4095) / 4096), b.ng), 256, 0, st>>>(d_lo, d_d24, d_blk, d_rg_start, d_blk_start, d_nblk, b.g0, d_pos, d_dev);
            if (grp_max[k]) k_check_span<<<dim3((unsigned)((grp_max[k] + 1023) / 1024), b.ng), 256, 0, st>>>(b);
        }
        k_tile_first<<<(unsigned)((nt_grp + 255) / 256), 256, 0, st>>>(a);
        k_cap_check<<<a.ng * chunks, 1024, 0, st>>>(a, chunks);
        k_tile_offsets<<<a.ng, 1024, 0, st>>>(a, d_rel, d_rg_words);
        k_pack_tiles<<<(unsigned)((nt_grp + 7) / 8), 256, 0, st>>>(a, w, 0);
        PD_CUDA(c, cudaGetLastError());
    }
    a.g0 = 0; a.ng = R;
    k_long_offsets<<<R, 1024, 0, st>>>(a, d_lcount, d_rg_longs);
    PD_CUDA(c, cudaGetLastError());
    std::vector<uint32_t> h_small((size_t)R + 16);
    std::vector<uint64_t> h_longs(R);
    PD_CUDA(c, cudaMemcpyAsync(h_small.data(), d_small, h_small.size() * 4, cudaMemcpyDeviceToHost, st));
    PD_CUDA(c, cudaMemcpyAsync(h_longs.data(), d_rg_longs, R * 8, cudaMemcpyDeviceToHost, st));
    PD_CUDA(c, cudaStreamSynchronize(st));
    if (h_small[2]) return pd_fail(c, PD_ERR_ARG, "pd_contig_push_pinned: position before the contig anchor");
    if (h_small[0]) return pd_fail(c, PD_ERR_ORDER, "pd_contig_push_pinned: read pairs must be sorted by position");
    bool fallback = h_small[1] != 0;
    for (uint32_t g = 0; g < R; ++g)
        if (c->rgc[g].max_load != 0xFFFFFFFFu && std::max(h_small[16 + g], c->rgc[g].lookback_tiles) > (uint32_t)CAP_MAX_LOOKBACK) fallback = true;
    if (fallback) return 1;

    if (ntile > c->cap_tiles || !c->d_tiles) {
        if (c->d_tiles) cudaFree(c->d_tiles);
        c->d_tiles = nullptr; c->cap_tiles = 0;
        size_t want = ntile + ntile / 8 + 64;
        PD_CUDA(c, cudaMalloc(&c->d_tiles, want * sizeof(PdTile)));
        c->cap_tiles = want;
    }
    w.tiles = c->d_tiles;
    std::vector<uint64_t> lbase(R + 1, 0);
    for (uint32_t g = 0; g < R; ++g) lbase[g + 1] = lbase[g] + h_longs[g];
    c->total_longs = lbase[R];
    if (c->total_longs > 0xFFFFFFF0ull) return pd_fail(c, PD_ERR_CAPACITY, "more than 2^32 long read pairs in one contig batch");
    c->h_long_off.assign(R + 1, 0);
    for (uint32_t g = 0; g <= R; ++g) c->h_long_off[g] = (uint32_t)lbase[g];
    PD_CUDA(c, cudaMemcpyAsync(d_long_base, lbase.data(), (R + 1) * 8, cudaMemcpyHostToDevice, st));
    if (c->total_longs + 1 > c->cap_longs || !c->d_longs) {
        if (c->d_longs) cudaFree(c->d_longs);
        c->d_longs = nullptr; c->cap_longs = 0;
        size_t want = c->total_longs + c->total_longs / 8 + 1024;
        PD_CUDA(c, cudaMalloc(&c->d_longs, want * sizeof(PdLong)));
        c->cap_longs = want;
    }
    if (grow_dev(c, 7, d_pmax, (size_t)c->total_longs + 1)) return c->status;
    w.longs = c->d_longs; w.pmax = d_pmax;
    k_pack_longs<<<(unsigned)((ntile + 255) / 256), 256, 0, st>>>(a, w);
    k_long_pmax<<<(R + 63) / 64, 64, 0, st>>>(a, w, d_rg_longs);
    k_tile_table<<<(unsigned)((ntile + 255) / 256), 256, 0, st>>>(a, w, d_rg_longs);
    PD_CUDA(c, cudaGetLastError());
    PD_CUDA(c, cudaEventRecord(c->ev[1], st));
    PD_CUDA(c, cudaStreamSynchronize(st));
    PD_CUDA(c, cudaEventElapsedTime(&c->ms_h2d, c->ev[0], c->ev[1]));
    return 0;
}
