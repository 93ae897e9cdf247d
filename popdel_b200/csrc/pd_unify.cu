// pd_unify.cu -- segment-level merge of the window calls ON THE DEVICE (SURVEY.md 8f rank 1).
//
// Reference: unifyCalls utils_popdel.h:567-654 with similar / delSizeSimilar / enoughOverlap / checkAndExtend
// (:237-320), lowerCall (:327-343), mergeWindowRange (:512-559), setGenotypes (:441-503), setFreqFromGTs (:344-366),
// called once per processSegment() (workflow_popdel.h:48). With pd_set_unify the scan keeps the window calls and
// their N x 13 per-sample rows in device memory and only the MERGED variants cross PCIe.
//
//   k_seg_bounds     window calls are emitted in window order, so the calls of one processSegment() are a run of equal
//                    `segment` tags: first / last index per segment.
//   k_unify_plan     one block per segment (merge loop: one warp in lockstep). All threads: stable rank sort by (position, deletion length, LR descending)
//                    and a working copy of the call headers in that order. Thread 0: the reference's merge loop -- a
//                    sequential state machine over a few dozen headers whose quirks must be kept (the running lists of
//                    starts / sizes and the window counters are only reset by a SUCCESSFUL mergeWindowRange, the first
//                    call of a later group is not in the lists, `last` itself is outside the merged range). It
//                    fixes position / length / LR / filter of every merged variant and lists its in-range windows.
//   k_unify_offsets  exclusive scan of the variants per segment -> output slots (segment order).
//   k_unify_list     output slot -> variant.
//   k_unify_emit     grid (variants, sample groups), one WARP per (variant, sample) with the lanes over the variant's
//                    in-range windows: PL sums -> setGenotypes, median LAD / DAD by bisection on the value over the
//                    column staged in shared memory, allele count -> frequency; header + row go to mapped host memory.
//   k_unify_freq     sample-sharded cohorts only: the plan depends on the call headers alone, which every rank holds
//                    identically, so every rank merges the same variants over its own samples' rows; the frequency then
//                    takes the allele counts of all ranks (all-gathered) over the cohort's n_global samples.
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "pd_device.cuh"
#include "pd_shard.h"

namespace {

struct UnifyArgs {
    const pd_call * calls; const uint32_t * ps;        // window calls of the scan (device), window order
    uint32_t n_raw, row_words, N, nseg;
    uint32_t n_global;                                 // samples of the cohort (sample-sharded: all ranks; else N)
    double sd, min_cover; int output_failed;
    int force_global;                                  // test knob (PD_UNIFY_GLOBAL): run the merge loop on global memory
    uint32_t * seg_first, * seg_last;                  // [nseg]
    uint32_t * seg_keep;                               // [nseg + 1] variants per segment, then their exclusive prefix
    // per window call; a segment owns the entries [seg_first, seg_last) of each array
    uint32_t * order;                                  // sorted slot -> index of the window call
    pd_call * wc;                                      // working copy of the headers in sorted order
    uint32_t * starts, * sizes;                        // the merge loop's running lists (append-only, "clear" = new offset)
    uint32_t * inr;                                    // window calls in range of the variant starting at a sorted slot
    uint32_t * gwc, * sig;                             // per sorted slot: in-range windows / significant windows (0: no merge)
    uint32_t * vlist;                                  // output slot -> sorted slot of the variant
    uint32_t * alleles, * blocks_done;                 // per output slot
    uint32_t * total;                                  // mapped host: number of variants
    pd_call * out_calls; uint32_t * out_ps; uint32_t * out_sig;     // mapped host
};

__device__ __forceinline__ bool all_pass(const pd_call & c) { return (c.filter & 31u) == 0; }        // :207-214

__device__ __forceinline__ bool size_similar(uint32_t a, uint32_t b, double sd)                      // :237-257
{
    const uint32_t l = min(a, b), r = max(a, b);
    return (l + 2 * sd >= r) || (l >= 0.5 * r);
}
// :306-320; may extend a.end_position (checkAndExtend :269-280)
__device__ __forceinline__ bool similar_calls(pd_call & a, const pd_call & b, double sd)
{
    if (!size_similar(a.deletion_length, b.deletion_length, sd)) return false;
    const uint32_t aSpan = a.end_position - a.position, bSpan = b.end_position - b.position;
    const uint32_t minLen = min(aSpan, bSpan);
    const uint32_t left = max(a.position, b.position), right = min(a.position + aSpan, b.position + bSpan);
    const int overlap = (int)(right - left);
    if (overlap >= 0.25 * minLen || overlap + 2 * sd >= minLen) return true;
    if ((aSpan < a.deletion_length || bSpan < b.deletion_length) &&
        (b.position - a.position < (min(a.deletion_length, b.deletion_length) + 4 * sd))) { a.end_position = b.end_position; return true; }
    return false;
}

__global__ void k_seg_bounds(UnifyArgs u)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= u.n_raw) return;
    const uint32_t s = u.calls[i].segment;
    if (s >= u.nseg) return;
    if (i == 0 || u.calls[i - 1].segment != s) u.seg_first[s] = i;
    if (i == u.n_raw - 1 || u.calls[i + 1].segment != s) u.seg_last[s] = i + 1;
}

constexpr uint32_t PLAN_CAP = 512;
__device__ __forceinline__ void plan_segment(const UnifyArgs & u, uint32_t seg, uint32_t n, pd_call * W, uint32_t * S, uint32_t * Z, uint32_t * I,
                             uint32_t * G, uint32_t * Q, const uint32_t * ord, int lane);

__global__ void __launch_bounds__(256) k_unify_plan(UnifyArgs u)
{
    const uint32_t seg = blockIdx.x, tid = threadIdx.x, T = blockDim.x;
    const uint32_t first = u.seg_first[seg], n = u.seg_last[seg] - first;
    if (n <= 1) { if (tid == 0) u.seg_keep[seg] = 0; return; }        // `calls.size() <= 1 -> false`: nothing is written
    // ---- std::sort by lowerCall; ties keep window order (the oracle's choice, equal keys are interchangeable headers)
    for (uint32_t i = tid; i < n; i += T) {
        const pd_call a = u.calls[first + i];
        uint32_t rank = 0;
        for (uint32_t j = 0; j < n; ++j) {
            const pd_call * b = u.calls + first + j;
            const uint32_t bp = __ldg(&b->position), bl = __ldg(&b->deletion_length);
            bool lower;
            if (bp != a.position) lower = bp < a.position;
            else if (bl != a.deletion_length) lower = bl < a.deletion_length;
            else { const double blr = __ldg(&b->lr); lower = blr > a.lr || (blr == a.lr && j < i); }
            rank += lower;
        }
        u.order[first + rank] = first + i;
        u.wc[first + rank] = a;
        u.gwc[first + rank] = 0; u.sig[first + rank] = 0;
    }
    __syncthreads();
    // the merge loop is sequential: run it on shared-memory copies when the segment fits (it nearly always does), so that
    // its few hundred dependent accesses cost shared-memory instead of L2 latency
    __shared__ pd_call s_w[PLAN_CAP];
    __shared__ uint32_t s_s[PLAN_CAP], s_z[PLAN_CAP], s_i[PLAN_CAP], s_g[PLAN_CAP], s_q[PLAN_CAP], s_o[PLAN_CAP];
    const bool fits = n <= PLAN_CAP && !u.force_global;
    if (fits) {
        for (uint32_t i = tid; i < n; i += T) { s_w[i] = u.wc[first + i]; s_o[i] = u.order[first + i]; s_g[i] = 0; s_q[i] = 0; }
        __syncthreads();
    }
    if (tid < 32) plan_segment(u, seg, n, fits ? s_w : u.wc + first, fits ? s_s : u.starts + first, fits ? s_z : u.sizes + first,
                               fits ? s_i : u.inr + first, fits ? s_g : u.gwc + first, fits ? s_q : u.sig + first, fits ? s_o : u.order + first, (int)tid);
    if (fits) {
        __syncthreads();
        for (uint32_t i = tid; i < n; i += T) {
            u.wc[first + i] = s_w[i]; u.inr[first + i] = s_i[i]; u.gwc[first + i] = s_g[i]; u.sig[first + i] = s_q[i]; u.starts[first + i] = s_s[i];
        }
    }
}

// value of rank k (0-based, ascending) of v[0, n): bisection on the value with warp-wide counts (v is not reordered)
__device__ __forceinline__ uint32_t warp_select_rank(const uint32_t * v, uint32_t n, uint32_t k, int lane)
{
    uint32_t lo = 0xFFFFFFFFu, hi = 0;
    for (uint32_t i = lane; i < n; i += 32) { const uint32_t x = v[i]; lo = min(lo, x); hi = max(hi, x); }
    lo = __reduce_min_sync(PD_FULL, lo); hi = __reduce_max_sync(PD_FULL, hi);
    while (lo < hi) {                                                  // smallest x with #{v <= x} >= k + 1
        const uint32_t mid = lo + (hi - lo) / 2;
        uint32_t c = 0;
        for (uint32_t i = lane; i < n; i += 32) c += v[i] <= mid;
        c = __reduce_add_sync(PD_FULL, c);
        if (c >= k + 1) hi = mid; else lo = mid + 1;
    }
    return lo;
}

// The reference's merge loop over the sorted headers W[0, n) of one segment, run by ONE WARP in lockstep: every lane walks
// the same sequential loop on the same values (the longest segment of the contig sets the kernel's time, and that time is
// a chain of dependent shared-memory accesses), lane 0 does the stores, and the two parts that are not sequential -- the
// medians of the running start / size lists (select by bisection, a few hundred entries for a long deletion) and the list
// of in-range windows of a merged variant -- use all 32 lanes.
__device__ __forceinline__ void plan_segment(const UnifyArgs & u, uint32_t seg, uint32_t n, pd_call * W, uint32_t * S, uint32_t * Z, uint32_t * I,
                             uint32_t * G, uint32_t * Q, const uint32_t * ord, int lane)
{
    const uint32_t last = n - 1;
    const uint32_t lt = (1u << lane) - 1u;
    uint32_t cur = 0;
    auto drop_all = [&]() { if (lane == 0) u.seg_keep[seg] = 0; };
    if (!u.output_failed) {
        while (!all_pass(W[cur])) { if (cur == last) { drop_all(); return; } ++cur; }
        if (cur == last) { drop_all(); return; }
    }
    const uint32_t first_idx = cur;
    for (uint32_t k = lane; k < first_idx; k += 32) W[k].filter = 255;
    uint32_t loff = 0, ln = 0;                                         // running lists = S/Z[loff, loff + ln)
    if (lane == 0) { S[0] = W[cur].position; Z[0] = W[cur].deletion_length; }
    ln = 1;
    double lr = W[cur].lr;                                             // (long double in the reference)
    uint32_t winCount = 1, sigWin = 1;
    __syncwarp();
    auto merge_range = [&](uint32_t start, uint32_t lastx) {           // mergeWindowRange :512-559 without the per-sample part
        __syncwarp();                                                  // (lane 0's appends to the lists)
        pd_call & st = W[start];
        const uint32_t mp = warp_select_rank(S + loff, ln, ln / 2, lane), ml = warp_select_rank(Z + loff, ln, ln / 2, lane);
        if (lane == 0) { st.position = mp; st.deletion_length = ml; st.lr = lr / winCount; }
        loff += ln; ln = 0;
        uint32_t g = 0;
        for (uint32_t k0 = start; k0 < lastx; k0 += 32) {              // in-range windows, in sorted order
            const uint32_t k = k0 + lane;
            bool in = false;
            if (k < lastx) { const uint32_t wp = W[k].window_position; in = wp > mp && wp - 30 < mp + ml; }
            const uint32_t bm = __ballot_sync(PD_FULL, in);
            if (in) I[start + g + __popc(bm & lt)] = ord[k];
            g += __popc(bm);
        }
        if (g == 0) { if (lane == 0) st.filter = 255; __syncwarp(); return; }      // (returns before the counters are reset)
        if (lane == 0) {
            G[start] = g; Q[start] = sigWin;
            if (30.0 * sigWin / ml < u.min_cover) st.filter |= 16;
        }
        __syncwarp();
        winCount = 1; sigWin = 1; lr = 0.0;
    };
    uint32_t it = first_idx + 1;
    // the three fields of W[cur] the comparison reads live in registers, W[it] is read once, W[it + 1] is in flight while W[it]
    // is compared
    pd_call a;
    a.position = W[cur].position; a.end_position = W[cur].end_position; a.deletion_length = W[cur].deletion_length;
    pd_call x = W[it];
    while (true) {
        pd_call nx = x;
        if (it != last) nx = W[it + 1];
        const uint32_t end_before = a.end_position;
        const bool similar = similar_calls(a, x, u.sd);
        if (a.end_position != end_before && lane == 0) W[cur].end_position = a.end_position;      // checkAndExtend
        if (similar) {
            if (all_pass(x)) { if (lane == 0) { S[loff + ln] = x.position; Z[loff + ln] = x.deletion_length; } ++ln; ++sigWin; }
            ++winCount;
            lr += x.lr;
            if (lane == 0) W[it].filter = 255;
            if (it == last) { if (ln) merge_range(cur, it); break; }
        } else {
            if (winCount != 1 && ln) merge_range(cur, it);
            else if (lane == 0) W[cur].filter = 255;
            cur = it;
            a.position = x.position; a.end_position = x.end_position; a.deletion_length = x.deletion_length;
        }
        if (it != last) { ++it; x = nx; }
        else { if (winCount == 1 && lane == 0) W[cur].filter = 255; break; }
    }
    __syncwarp();
    uint32_t keep = 0;                                                 // kept sorted slots, in order (the lists are no longer needed)
    for (uint32_t k0 = first_idx; k0 <= last; k0 += 32) {
        const uint32_t k = k0 + lane;
        const bool kp = k <= last && W[k].filter != 255;
        const uint32_t bm = __ballot_sync(PD_FULL, kp);
        if (kp) S[keep + __popc(bm & lt)] = k;
        keep += __popc(bm);
    }
    if (lane == 0) u.seg_keep[seg] = keep;
}

__global__ void __launch_bounds__(1024) k_unify_offsets(UnifyArgs u)
{
    __shared__ unsigned long long ws[33];
    unsigned long long carry = 0;
    for (uint32_t base = 0; base < u.nseg; base += blockDim.x) {
        const uint32_t i = base + threadIdx.x;
        const unsigned long long v = i < u.nseg ? u.seg_keep[i] : 0ull;
        unsigned long long tot;
        const unsigned long long ex = block_excl_scan(v, ws, tot);
        if (i < u.nseg) u.seg_keep[i] = (uint32_t)(carry + ex);
        carry += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) { u.seg_keep[u.nseg] = (uint32_t)carry; *u.total = (uint32_t)carry; }
}

// output slot -> sorted slot of its variant (segment order, then sorted order)
__global__ void k_unify_list(UnifyArgs u)
{
    const uint32_t seg = blockIdx.x * blockDim.x + threadIdx.x;
    if (seg >= u.nseg) return;
    uint32_t slot = u.seg_keep[seg];
    if (u.seg_keep[seg + 1] == slot) return;
    const uint32_t first = u.seg_first[seg], cnt = u.seg_keep[seg + 1] - slot;
    for (uint32_t i = 0; i < cnt; ++i) u.vlist[slot + i] = first + u.starts[first + i];         // kept sorted slots, left by k_unify_plan
}

constexpr int EMIT_WARPS_U = 8;
constexpr uint32_t EMIT_STAGE = 1024;                     // in-range windows whose values a warp stages in shared memory

// grid (variants, sample groups): one WARP per (variant, sample), lanes over the variant's in-range windows. Every value
// is read once per column; the medians are found by bisection on the value over the staged column (warp-wide counts).
__global__ void __launch_bounds__(EMIT_WARPS_U * 32) k_unify_emit(UnifyArgs u)
{
    __shared__ uint32_t s_vals[EMIT_WARPS_U][EMIT_STAGE];
    __shared__ uint32_t s_last;
    const uint32_t slot = blockIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t vs = u.vlist[slot];                            // sorted slot of this variant
    const pd_call hdr = u.wc[vs];
    const uint32_t g = u.gwc[vs];
    const uint32_t * own = u.ps + (size_t)u.order[vs] * u.row_words;
    const uint32_t * inr = u.inr + vs;
    uint32_t * orow = u.out_ps + (size_t)slot * u.row_words;
    uint32_t * vals = s_vals[wid];
    uint32_t alleles = 0;
    for (uint32_t s = blockIdx.y * EMIT_WARPS_U + wid; s < u.N; s += gridDim.y * EMIT_WARPS_U) {
        if (g == 0) {                                              // kept without a merge (stale counters at the end of the loop)
            if (lane < 13) orow[13 * s + lane] = own[13 * s + lane];
            continue;
        }
        // ---- setGenotypes :441-503: PL sums over the in-range windows
        uint32_t p0 = 0, p1 = 0, p2 = 0;
        for (uint32_t i = lane; i < g; i += 32) {
            const uint32_t * r = u.ps + (size_t)inr[i] * u.row_words + 13 * s;
            p0 += r[0]; p1 += r[1]; p2 += r[2];
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { p0 += __shfl_xor_sync(PD_FULL, p0, o); p1 += __shfl_xor_sync(PD_FULL, p1, o); p2 += __shfl_xor_sync(PD_FULL, p2, o); }
        const double mn = (double)min(min(p0, p1), p2);
        const double ref = (p0 - mn) / g, het = (p1 - mn) / g, hom = (p2 - mn) / g;
        uint32_t o0 = (uint32_t)round(ref), o1 = (uint32_t)round(het), o2 = (uint32_t)round(hom);
        // ---- median LAD / DAD: element g/2 of the sorted values, by bisection on the value
        uint32_t med = 0;                                          // lane j keeps the median of column j
        for (int j = 0; j < 8; ++j) {
            uint32_t lo = 0xFFFFFFFFu, hi = 0;
            for (uint32_t i = lane; i < g; i += 32) {
                const uint32_t v = u.ps[(size_t)inr[i] * u.row_words + 13 * s + 3 + j];
                if (i < EMIT_STAGE) vals[i] = v;
                lo = min(lo, v); hi = max(hi, v);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { lo = min(lo, __shfl_xor_sync(PD_FULL, lo, o)); hi = max(hi, __shfl_xor_sync(PD_FULL, hi, o)); }
            __syncwarp();
            const uint32_t need = g / 2 + 1;
            while (lo < hi) {
                const uint32_t mid = lo + (hi - lo) / 2;
                uint32_t cnt = 0;
                for (uint32_t i = lane; i < g; i += 32)
                    cnt += (i < EMIT_STAGE ? vals[i] : u.ps[(size_t)inr[i] * u.row_words + 13 * s + 3 + j]) <= mid;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(PD_FULL, cnt, o);
                if (cnt >= need) hi = mid; else lo = mid + 1;
            }
            if ((int)lane == j) med = lo;
            __syncwarp();
        }
        if (o1 == o2) { if (het > hom) ++o1; else ++o2; }
        else if (o0 == o1) { if (ref > het) ++o0; else ++o1; }
        if (o0 != 0) alleles += (o1 == 0) ? 1 : 2;                 // setFreqFromGTs :344-366 (counted by every lane alike)
        const uint32_t mcol = __shfl_sync(PD_FULL, med, (lane >= 3 && lane < 11) ? (int)lane - 3 : 0);
        uint32_t w = 0;
        if (lane == 0) w = o0; else if (lane == 1) w = o1; else if (lane == 2) w = o2;
        else if (lane < 11) w = mcol;
        else if (lane < 13) w = own[13 * s + lane];
        if (lane < 13) orow[13 * s + lane] = w;
    }
    // ---- allele count of the variant over all blocks of its row; the last block writes the header
    if (lane == 0 && alleles) atomicAdd(u.alleles + slot, alleles);
    __syncthreads();
    if (threadIdx.x == 0) { __threadfence(); s_last = atomicAdd(u.blocks_done + slot, 1u) == gridDim.y - 1; }
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        __threadfence();
        pd_call h = hdr;
        if (g) h.frequency = (double)atomicAdd(u.alleles + slot, 0u) / (u.N * 2.0);
        u.out_calls[slot] = h; u.out_sig[slot] = g ? u.sig[vs] : 0u;
    }
}

// parts = [world][total] allele counts of the ranks; the expression is that of k_unify_emit with the cohort's sample count
__global__ void k_unify_freq(UnifyArgs u, const uint32_t * __restrict__ parts, uint32_t total, uint32_t world)
{
    const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= total || u.gwc[u.vlist[slot]] == 0) return;      // kept without a merge: the window call's cohort frequency
    uint32_t a = 0;
    for (uint32_t r = 0; r < world; ++r) a += parts[(size_t)r * total + slot];
    u.out_calls[slot].frequency = (double)a / (u.n_global * 2.0);
}

template <typename T>
int grow(pd_ctx * c, int slot, T *& p, size_t need)
{
    const size_t bytes = std::max<size_t>(need, 1) * sizeof(T);
    if (bytes > c->cap_unify[slot] || !c->d_unify[slot]) {
        if (c->d_unify[slot]) cudaFree(c->d_unify[slot]);
        c->d_unify[slot] = nullptr; c->cap_unify[slot] = 0;
        const size_t want = std::max<size_t>(bytes + bytes / 4, 4096);
        PD_CUDA(c, cudaMalloc(&c->d_unify[slot], want));
        c->cap_unify[slot] = want;
    }
    p = reinterpret_cast<T *>(c->d_unify[slot]);
    return 0;
}

// sample-sharded: all-gathers the variant count of every rank; fails on every rank when they differ
int shard_agree_total(pd_ctx * c, uint32_t total)
{
    PdShard * s = c->shard;
    uint32_t all[PD_MAX_WORLD];
    PD_CUDA(c, cudaMemcpyAsync(s->d_small, &total, 4, cudaMemcpyHostToDevice, c->stream));
    if (pd_shard_allgather(c, s->d_small, (char *)s->d_small + 1024, 4, c->stream)) return c->status;
    PD_CUDA(c, cudaMemcpyAsync(all, (char *)s->d_small + 1024, 4 * s->world, cudaMemcpyDeviceToHost, c->stream));
    PD_CUDA(c, cudaStreamSynchronize(c->stream));
    for (uint32_t r = 0; r < s->world; ++r)
        if (all[r] != total) return pd_fail(c, PD_ERR_ARG, "sample-sharded scan: ranks disagree on the merged variants");
    return 0;
}

}  // namespace

// device-side buffers of the window calls (unify mode): grown so that `need_calls` fit; the first `keep_calls` survive
int pd_unify_ensure_raw(pd_ctx * c, size_t need_calls, size_t row, size_t keep_calls)
{
    if (need_calls > c->cap_u_calls || !c->d_u_calls) {
        const size_t floor_calls = getenv("PD_UNIFY_CAP") ? (size_t)std::max(1, atoi(getenv("PD_UNIFY_CAP"))) : 1024;      // test knob
        const size_t want = std::max<size_t>(need_calls + need_calls / 2, floor_calls);
        pd_call * p = nullptr;
        PD_CUDA(c, cudaMalloc(&p, want * sizeof(pd_call)));
        if (keep_calls) PD_CUDA(c, cudaMemcpy(p, c->d_u_calls, keep_calls * sizeof(pd_call), cudaMemcpyDeviceToDevice));
        cudaFree(c->d_u_calls);
        c->d_u_calls = p; c->cap_u_calls = want;
    }
    if (need_calls * row > c->cap_u_ps || !c->d_u_ps) {
        const size_t want = std::max<size_t>((need_calls + need_calls / 2) * row, getenv("PD_UNIFY_CAP") ? 64 : 1u << 18);
        uint32_t * p = nullptr;
        if (cudaMalloc(&p, want * 4) != cudaSuccess) {
            cudaGetLastError();
            return pd_fail(c, PD_ERR_CAPACITY, "device-side unify: the window calls of this scan do not fit device memory; scan a smaller window range");
        }
        if (keep_calls) PD_CUDA(c, cudaMemcpy(p, c->d_u_ps, keep_calls * row * 4, cudaMemcpyDeviceToDevice));
        cudaFree(c->d_u_ps);
        c->d_u_ps = p; c->cap_u_ps = want;
    }
    return 0;
}

void pd_unify_release(pd_ctx * c)
{
    cudaFree(c->d_u_calls); cudaFree(c->d_u_ps);
    for (auto & p : c->d_unify) cudaFree(p);
    if (c->res_sig) cudaFreeHost(c->res_sig);
}

// merges the n_raw window calls held in d_u_calls / d_u_ps; variants go to res_calls / res_ps / res_sig (mapped host)
int pd_run_unify(pd_ctx * c, uint32_t n_raw, size_t row, uint32_t nseg, int (*ensure_results)(pd_ctx *, size_t, size_t, size_t),
                 uint64_t * n_out, uint64_t * launches)
{
    *n_out = 0;
    PdShard * sh = c->shard;
    if (n_raw == 0 && !sh) return 0;
    cudaStream_t st = c->stream;
    UnifyArgs u;
    memset(&u, 0, sizeof(u));
    u.calls = c->d_u_calls; u.ps = c->d_u_ps; u.n_raw = n_raw; u.row_words = (uint32_t)row; u.N = c->N; u.nseg = nseg;
    u.n_global = sh ? sh->n_global : c->N;
    u.force_global = getenv("PD_UNIFY_GLOBAL") != nullptr;
    u.sd = c->unify.mean_stddev; u.min_cover = c->unify.min_relative_window_cover; u.output_failed = c->unify.output_failed;
    // (sample-sharded: this stage starts after the rank's last EM chunk has completed, and that chunk only completes once
    // every peer's last EM launch is running and has posted its statistics; no peer kernel waits for this rank any more, so
    // the allocations below may synchronise the device -- the rule of pd_shard_prelaunch does not apply here)
    if (n_raw) {
        if (grow(c, 0, u.seg_first, (size_t)nseg)) return c->status;
        if (grow(c, 1, u.seg_last, (size_t)nseg)) return c->status;
        if (grow(c, 2, u.seg_keep, (size_t)nseg + 1)) return c->status;
        if (grow(c, 3, u.order, (size_t)n_raw)) return c->status;
        if (grow(c, 4, u.wc, (size_t)n_raw)) return c->status;
        if (grow(c, 5, u.starts, (size_t)n_raw)) return c->status;
        if (grow(c, 6, u.sizes, (size_t)n_raw)) return c->status;
        if (grow(c, 7, u.inr, (size_t)n_raw)) return c->status;
        if (grow(c, 8, u.gwc, (size_t)n_raw)) return c->status;
        if (grow(c, 9, u.sig, (size_t)n_raw)) return c->status;
        u.total = c->res_count + 1;
        PD_CUDA(c, cudaMemsetAsync(u.seg_first, 0, (size_t)nseg * 4, st));
        PD_CUDA(c, cudaMemsetAsync(u.seg_last, 0, (size_t)nseg * 4, st));
        k_seg_bounds<<<(n_raw + 255) / 256, 256, 0, st>>>(u);
        k_unify_plan<<<nseg, 256, 0, st>>>(u);
        k_unify_offsets<<<1, 1024, 0, st>>>(u);
        *launches += 3;
        PD_CUDA(c, cudaGetLastError());
        PD_CUDA(c, cudaStreamSynchronize(st));
    }
    const uint32_t total = n_raw ? c->res_count[1] : 0;
    // every rank must enter the same exchanges: the plan depends on the (identical) call headers only, so the counts agree;
    // if they do not, every rank fails here instead of some of them waiting for the allele exchange below
    if (sh && shard_agree_total(c, total)) return c->status;
    if (total) {
        if (ensure_results(c, total, row, 0)) return c->status;
        if (total > c->cap_res_sig || !c->res_sig) {
            if (c->res_sig) cudaFreeHost(c->res_sig);
            c->res_sig = nullptr; c->cap_res_sig = 0;
            const size_t want = std::max<size_t>((size_t)total + total / 2, 1024);
            PD_CUDA(c, cudaHostAlloc(&c->res_sig, want * 4, cudaHostAllocMapped));
            c->cap_res_sig = want;
        }
        u.out_calls = c->res_calls; u.out_ps = c->res_ps; u.out_sig = c->res_sig;
        if (grow(c, 10, u.vlist, (size_t)total)) return c->status;
        if (grow(c, 11, u.alleles, (size_t)total)) return c->status;
        if (grow(c, 12, u.blocks_done, (size_t)total)) return c->status;
        PD_CUDA(c, cudaMemsetAsync(u.alleles, 0, (size_t)total * 4, st));
        PD_CUDA(c, cudaMemsetAsync(u.blocks_done, 0, (size_t)total * 4, st));
        k_unify_list<<<(nseg + 127) / 128, 128, 0, st>>>(u);
        // enough blocks per variant to occupy the GPU even when a scan yields few variants
        const uint32_t per_row = (c->N + EMIT_WARPS_U - 1) / EMIT_WARPS_U;
        const uint32_t gy = std::max<uint32_t>(1, std::min<uint32_t>(per_row, (4 * 148 + total - 1) / total));
        k_unify_emit<<<dim3(total, gy), EMIT_WARPS_U * 32, 0, st>>>(u);
        *launches += 2;
        PD_CUDA(c, cudaGetLastError());
        if (sh) {                                                 // allele counts of every rank -> the cohort's frequency
            const size_t need = (size_t)total * 4 * sh->world;
            if (need > sh->cap_recv) {
                cudaFree(sh->d_recv); sh->d_recv = nullptr; sh->cap_recv = 0;
                PD_CUDA(c, cudaMalloc(&sh->d_recv, need + need / 4)); sh->cap_recv = need + need / 4;
            }
            if (pd_shard_allgather(c, u.alleles, sh->d_recv, (size_t)total * 4, st)) return c->status;
            k_unify_freq<<<(total + 255) / 256, 256, 0, st>>>(u, (const uint32_t *)sh->d_recv, total, sh->world);
            *launches += 1;
            PD_CUDA(c, cudaGetLastError());
        }
        PD_CUDA(c, cudaStreamSynchronize(st));
    }
    *n_out = total;
    return 0;
}
