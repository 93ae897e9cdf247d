// pd_em2.cu -- K3-K5, second generation: the genotyping of every (window, initial length) pair as a BULK-SYNCHRONOUS,
// SAMPLE-MAJOR pipeline (replaces the pair-major kernels of pd_em.cu for cohorts that are not sharded by sample).
//
// Why: the pair-major kernels gather one 32-byte likelihood-table row per read pair and pass from tables that only
// fit L2 (100 read groups x 302 rows x 64 B); every lane of a warp belongs to another read group, so every gather is
// its own L1 wavefront (~2 cycles each, profiles/r02/em_stats_k_em_one_baseline.json: 4.7 cycles per gather measured).
// Here a block owns ONE read group: its table (32 B per row for the EM, 24 B for the final pass) is staged in
// shared memory once per block and the gathers become shared-memory loads.
//
//   k_e2_prep         per (read group, group of 2048 pairs): counting sort of the group's items (pair, read group) by
//                     (carrier of the initial length, number of active read pairs), so that the 32 lanes of a warp get
//                     items of equal length and the items that need later passes share warps; copies the items'
//                     deviations / positions from the window-major pool into a lane-interleaved layout [j][lane].
//   k_e2_reads<A>     sample-major data-likelihood pass (compute_data_likelihoods, EM overload,
//                     genotype_deletion_popdel_call.h:179-253): lane = item, sums ln ref / ln((ref+del)/2) / ln del and
//                     the posterior-weight moments sum r, sum r*d (r = del/(del+ref)) in read-pair order. Pass A (initial
//                     length, zero shifts) also counts initialize_allele_frequency's window (:93-133). An item is only
//                     recomputed when its reference shift changed or it carries read pairs inside the deletion
//                     hypothesis' histogram at the old or the new length.
//   k_e2_pair         pair-major, one block per pair: per-sample triples (finish_triple), allele frequency
//                     (:467-485), convergence test and the partial "previous state" comparison (:598-660), length and
//                     reference-shift update from the moments (:388-462, rgDlIt quirk), requests the next pass.
//   k_e2_final_reads  sample-major final pass (:255-337 without the ln sums, which equal the last EM pass): log10
//                     likelihood sums, LAD, DAD (:137-172), first/last positions, supporting read pairs.
//   k_e2_final_pair   per surviving pair: PL (utils_popdel.h:1511-1528), percentiles of the supporting read pairs
//                     (:514-529), likelihood ratio (:490-508), the Call.
// Control flow between the kernels travels in device memory (per-item control words, per-pair state); the host
// enqueues the fixed sequence prep, A, pair, (reads, pair) x (iterations + 1), final_reads, final_pair without
// synchronising; blocks without work exit at once.
#include <algorithm>
#include <cstdio>
#include <cstdlib>

#include "pd_em_common.cuh"

#ifdef PD_EM_STATS
__device__ unsigned long long g_e2_stats[32];
#define S2_ADD(i, v) atomicAdd(&g_e2_stats[i], (unsigned long long)(v))
extern "C" int pd_debug_e2_stats(unsigned long long * out)
{
    unsigned long long z[32] = {};
    if (cudaMemcpyFromSymbol(out, g_e2_stats, sizeof(z)) != cudaSuccess) return -1;
    if (cudaMemcpyToSymbol(g_e2_stats, z, sizeof(z)) != cudaSuccess) return -1;
    return 0;
}
#else
#define S2_ADD(i, v) do {} while (0)
#endif

namespace {

constexpr int E2_SUB = 1024;                       // pairs per sort group
constexpr int E2_WBS = E2_SUB / 32;                // warp blocks per sort group
constexpr int E2_T = 256;
#ifndef E2_MINB
#define E2_MINB 3
#endif
constexpr uint32_t E2_LMASK = (1u << 30) - 1;
enum { E2_NONE = 0, E2_M1 = 1, E2_M2 = 2, E2_FIN = 3 };
enum { PH_A = 0, PH_M1 = 1, PH_M2 = 2, PH_ALIVE = 3, PH_DEAD = 4, PH_DONE = 5 };
constexpr uint32_t E2_SUPP_CAP = 1536;             // supporting read pairs kept per pair for the percentiles

struct E2Item { uint32_t off; uint32_t n; int32_t dmx; uint32_t pair; };             // sorted-major, static
struct E2Ctl { int32_t shift; uint32_t lmode; int32_t supp_lo, supp_hi; };           // sorted-major, written by k_e2_pair
struct E2Cur { int32_t Lc, Sc, LcA, pad; };                                          // what rec / recA were computed with
// pair-major [pair][rg], 64 bytes = two sectors, moved with 128-bit accesses. sd / c (sum of deviations, window count
// of initialize_allele_frequency :93-133) are only meaningful in the records of pass A (recA).
struct alignas(16) E2Rec { double l0, l1, l2, sr, srd; uint32_t nd; uint32_t c; int32_t sd; uint32_t pad[3]; };
struct alignas(16) E2Fin { double t0, t1, t2; uint32_t lad[3], dad[5], fl_min, fl_max, nsupp, pad[3]; };
static_assert(sizeof(E2Rec) == 64 && sizeof(E2Fin) == 80, "record sizes");

template <typename R>
__device__ __forceinline__ void rec_store(R * dst, const R & r)
{
    const uint4 * s4 = reinterpret_cast<const uint4 *>(&r);
    uint4 * d4 = reinterpret_cast<uint4 *>(dst);
#pragma unroll
    for (int i = 0; i < (int)(sizeof(R) / 16); ++i) d4[i] = s4[i];
}
template <typename R>
__device__ __forceinline__ R rec_load(const R * src)
{
    R r;
    uint4 * d4 = reinterpret_cast<uint4 *>(&r);
    const uint4 * s4 = reinterpret_cast<const uint4 *>(src);
#pragma unroll
    for (int i = 0; i < (int)(sizeof(R) / 16); ++i) d4[i] = s4[i];
    return r;
}
struct E2Pair {
    int32_t L0; uint32_t len, it, prev_len, phase, nvisited, src_a, pad;
    double freq, prev_freq, lr_conv, gt[3];
    int32_t vlen[64]; double vfreq[64];
};

struct E2Args {
    E2Item * item; E2Ctl * ctl; E2Cur * cur;         // [groups * E2_SUB]
    E2Rec * rec, * recA; uint32_t * inv; E2Fin * fin;      // [pairs * R]
    E2Pair * pst;                                    // [pairs]
    uint32_t * blk_off; uint32_t * blk_nmax;         // [groups * E2_WBS] slab of the warp block (words) / its longest item
    uint32_t * wbflag, * finflag;                    // [groups * E2_WBS] pass number that has work for the warp block / final pass
    int32_t * devT; uint32_t * posT; uint32_t devt_cap;      // lane-interleaved copies of the items' read pairs: [j / 4][lane][4]
    uint32_t * devt_used;                            // device counter (words)
    uint32_t * ovf;                                  // set when devT is too small (the scan is repeated with more room)
    uint32_t * suppn; uint32_t * supp_first, * supp_last;     // [pairs], [pairs * E2_SUPP_CAP]
    uint32_t * act;                                  // [3][pairs] pairs that asked for the next pass (rotating lists)
    uint32_t * actn;                                 // [3] their counts, [3] = surviving pairs
    uint32_t * alive;                                // [pairs] surviving pairs (final pass)
    uint32_t nsub, npairs;
};

// shared-memory loads by 32-bit shared-window address (the tables are read-only after the staging barrier)
__device__ __forceinline__ double2 lds_d2(uint32_t addr)
{
    double2 v;
    asm("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ double lds_d(uint32_t addr)
{
    double v;
    asm("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}

__device__ __forceinline__ void st_release_gpu(uint32_t * p, uint32_t v)
{
    asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}

// ------------------------------------------------------------------------------------------------------------------
// prep
// ------------------------------------------------------------------------------------------------------------------
constexpr int E2_IPT = E2_SUB / E2_T;               // items per thread in k_e2_prep

__global__ void __launch_bounds__(E2_T) k_e2_prep(PdDev a, EmArgs e, E2Args x)
{
    __shared__ uint32_t s_hist[264], s_start[264];
    __shared__ uint32_t s_n[E2_SUB], s_off[E2_SUB];
    __shared__ uint32_t s_nmax[E2_WBS], s_boff[E2_WBS];
    __shared__ uint32_t s_base;
    __shared__ unsigned long long s_ws[33];
    __shared__ uint32_t s_tile[E2_T / 32][32 * 33];
    const uint32_t tid = threadIdx.x, sub = blockIdx.x, g = pd_grid_row();
    if (g >= a.R) return;
    const uint32_t p_lo = sub * E2_SUB, np = min((uint32_t)E2_SUB, e.npairs - p_lo);
    const uint32_t grp = g * x.nsub + sub;
    const size_t sbase = (size_t)grp * E2_SUB;
    const PdRgConst * rg = a.rgc + g;
    const uint32_t max_load = __ldg(&rg->max_load), smp = __ldg(&rg->sample);
    const int hb = __ldg(&rg->hist_base);
    for (uint32_t i = tid; i < 264; i += E2_T) s_hist[i] = 0;
    for (uint32_t i = tid; i < (uint32_t)E2_SUB; i += E2_T) s_n[i] = 0;
    __syncthreads();
    // ---- keys (the item's inputs stay in registers for the scatter)
    uint32_t v_n[E2_IPT], v_off[E2_IPT], v_key[E2_IPT], v_rank[E2_IPT]; int32_t v_dmx[E2_IPT], v_L0[E2_IPT];
    {
        uint32_t v_job[E2_IPT], v_cj[E2_IPT];
#pragma unroll
        for (int k = 0; k < E2_IPT; ++k) {
            const uint32_t i = tid + k * E2_T;
            v_L0[k] = 0; v_job[k] = 0;
            if (i < np) { const PdPair pr = e.pairs[e.pair0 + p_lo + i]; v_L0[k] = pr.L0; v_job[k] = pr.job - e.job_base; }
        }
#pragma unroll
        for (int k = 0; k < E2_IPT; ++k) v_cj[k] = (tid + k * E2_T < np) ? e.cjob_of[v_job[k]] - e.cj_base : 0u;
#pragma unroll
        for (int k = 0; k < E2_IPT; ++k) {
            const bool ok = tid + k * E2_T < np;
            v_n[k] = ok ? e.act_cnt[(size_t)v_cj[k] * a.R + g] : 0u;
            v_off[k] = ok ? e.act_off[(size_t)v_cj[k] * a.R + g] : 0u;
            v_dmx[k] = ok ? e.dmax[(size_t)v_job[k] * a.N + smp] : INT_MIN;
        }
    }
#pragma unroll
    for (int k = 0; k < E2_IPT; ++k) {
        const uint32_t i = tid + k * E2_T;
        if (i >= np) continue;
        const uint32_t n = v_n[k];
        uint32_t key;
        if (n == 0 || n >= max_load) { key = 256; v_n[k] = 0; }
        else key = (v_dmx[k] >= v_L0[k] - hb + 1 ? 0u : 128u) + (127u - min(n, 127u));
        v_key[k] = key;
        v_rank[k] = atomicAdd(&s_hist[key], 1u);
        if (g == 0) {                                            // per-pair state is initialised by the blocks of read group 0
            E2Pair & st = x.pst[p_lo + i];
            st.L0 = v_L0[k]; st.len = (uint32_t)v_L0[k]; st.it = 0; st.prev_len = (uint32_t)v_L0[k]; st.phase = PH_A; st.nvisited = 0; st.src_a = 0;
            st.freq = 0; st.prev_freq = 0; st.lr_conv = 0;
        }
    }
    __syncthreads();
    {
        static_assert(E2_T == 256, "one thread per key bin");
        unsigned long long total;
        const unsigned long long ex = block_excl_scan((unsigned long long)s_hist[tid], s_ws, total);
        s_start[tid] = (uint32_t)ex;
        if (tid == 0) s_start[256] = (uint32_t)total;                       // empty / high-coverage items go last
    }
    __syncthreads();
    // ---- scatter into sorted order
#pragma unroll
    for (int k = 0; k < E2_IPT; ++k) {
        const uint32_t i = tid + k * E2_T;
        if (i >= np) continue;
        const uint32_t p = p_lo + i;
        const uint32_t slot = s_start[v_key[k]] + v_rank[k];
        x.item[sbase + slot] = E2Item{v_off[k], v_n[k], v_dmx[k], p};
        x.ctl[sbase + slot] = E2Ctl{0, (uint32_t)v_L0[k] & E2_LMASK, 0, 0};
        x.cur[sbase + slot] = E2Cur{INT_MIN, 0, v_L0[k], 0};
        x.inv[(size_t)p * a.R + g] = (uint32_t)(sbase + slot);
        s_n[slot] = v_n[k]; s_off[slot] = v_off[k];
    }
    for (uint32_t i = np + tid; i < (uint32_t)E2_SUB; i += E2_T) {              // padding slots of the last group
        x.item[sbase + i] = E2Item{0, 0, INT_MIN, 0xFFFFFFFFu};
        x.ctl[sbase + i] = E2Ctl{0, 0, 0, 0};
    }
    __syncthreads();
    // ---- warp blocks: longest item, slab offsets (32 lanes x the longest item rounded up to 4 read pairs)
    if (tid < (uint32_t)E2_WBS) {
        uint32_t m = 0;
        for (int k = 0; k < 32; ++k) m = max(m, s_n[tid * 32 + ((k + tid) & 31)]);
        s_nmax[tid] = m;
    }
    __syncthreads();
    if (tid == 0) {
        uint32_t tot = 0;
        for (int w = 0; w < E2_WBS; ++w) { s_boff[w] = tot; tot += 32u * ((s_nmax[w] + 3u) & ~3u); }
        uint32_t base = tot ? atomicAdd(x.devt_used, tot) : 0u;
        if ((uint64_t)base + tot > x.devt_cap) { atomicExch(x.ovf, 1u); base = 0xFFFFFFFFu; }
        s_base = base;
    }
    __syncthreads();
    const uint32_t base = s_base;
    if (tid < (uint32_t)E2_WBS) {
        x.blk_off[(size_t)grp * E2_WBS + tid] = base == 0xFFFFFFFFu ? 0u : base + s_boff[tid];
        x.blk_nmax[(size_t)grp * E2_WBS + tid] = base == 0xFFFFFFFFu ? 0u : s_nmax[tid];
        x.wbflag[(size_t)grp * E2_WBS + tid] = 0; x.finflag[(size_t)grp * E2_WBS + tid] = 0;
    }
    if (base == 0xFFFFFFFFu) return;
    // ---- copy the read pairs through a shared-memory tile: rows are read along the pool (one item per warp load, 8 loads
    // in flight), columns are written lane-interleaved, 4 read pairs of one item per 128-bit store. Within every run of
    // 32 read pairs those ABOVE the reference histogram (the only ones that can fall inside the histogram of a deletion
    // hypothesis) are moved to the front, so that the rare path of the likelihood passes is left early by the whole warp.
    const uint32_t lane = tid & 31, warp = tid >> 5;
    uint32_t * tile = s_tile[warp];
    const int hi_dev = (int)__ldg(&rg->hist_len) - 2 - (hb - 1);           // deviations >= hi_dev lie above the histogram
    const uint32_t lt = (1u << lane) - 1u;
    for (uint32_t wb = warp; wb < (uint32_t)E2_WBS; wb += E2_T / 32) {
        const uint32_t nmax = s_nmax[wb];
        if (nmax == 0) continue;
        const uint32_t npad = (nmax + 3u) & ~3u;
        const uint32_t my_n = s_n[wb * 32 + lane], my_off = s_off[wb * 32 + lane];
        const size_t slab = (size_t)base + s_boff[wb];
        for (uint32_t c0 = 0; c0 < npad; c0 += 32) {
            const uint32_t j = c0 + lane;
            const uint32_t jend = min(npad - c0, 32u);
            uint32_t bal[32];
            for (int arr = 0; arr < 2; ++arr) {
                const uint32_t * src = arr ? e.pool_pos : reinterpret_cast<const uint32_t *>(e.pool_dev);
                uint32_t * dst = arr ? x.posT : reinterpret_cast<uint32_t *>(x.devT);
                __syncwarp();
#pragma unroll
                for (uint32_t i0 = 0; i0 < 32; i0 += 8) {
                    uint32_t v[8];
#pragma unroll
                    for (uint32_t k = 0; k < 8; ++k) {
                        const uint32_t n_i = __shfl_sync(PD_FULL, my_n, (int)(i0 + k)), o_i = __shfl_sync(PD_FULL, my_off, (int)(i0 + k));
                        v[k] = j < n_i ? __ldg(src + o_i + j) : 0u;
                    }
#pragma unroll
                    for (uint32_t k = 0; k < 8; ++k) {
                        const uint32_t n_i = __shfl_sync(PD_FULL, my_n, (int)(i0 + k));
                        const bool valid = j < n_i;
                        if (arr == 0) bal[i0 + k] = __ballot_sync(PD_FULL, valid && (int)v[k] >= hi_dev);
                        const uint32_t m = bal[i0 + k], vm = __ballot_sync(PD_FULL, valid);
                        const uint32_t pos = !valid ? lane : ((m >> lane) & 1u ? __popc(m & lt) : __popc(m) + __popc(vm & ~m & lt));
                        tile[(i0 + k) * 33 + pos] = v[k];
                    }
                }
                __syncwarp();
                for (uint32_t jj = 0; jj < jend; jj += 4) {
                    const uint4 v = make_uint4(tile[lane * 33 + jj], tile[lane * 33 + jj + 1], tile[lane * 33 + jj + 2], tile[lane * 33 + jj + 3]);
                    *reinterpret_cast<uint4 *>(dst + slab + (size_t)((c0 + jj) >> 2) * 128 + lane * 4) = v;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// data-likelihood pass
// ------------------------------------------------------------------------------------------------------------------
// Shared-memory image of the read group's table for the EM passes, 32 B per row in three arrays:
//   sA[r] = {ln val, g1b}   g1b = ln(val + floor) - ln 2, or ln val for rows ON the floor (val == min_prob)
//   sR[r] = rbs             floor / (floor + val), or -0.5 for rows on the floor (sign = "counts as ref == del")
//   sV[r] = val             only read when the deletion hypothesis is inside the histogram
// so that the bulk of the read pairs (deletion hypothesis on the floor) needs no comparison of likelihood values:
// g1 = g1b, r = |rbs|, nd += rbs < 0  (compute_data_likelihoods :179-253 with the look-ups of pd_em.cu's dl_one).
template <bool PASS_A>
__global__ void __launch_bounds__(E2_T, E2_MINB) k_e2_reads(PdDev a, EmArgs e, E2Args x, uint32_t pass_no)
{
    extern __shared__ double2 s_tab[];
    const uint32_t tid = threadIdx.x, sub = blockIdx.x, g = pd_grid_row();
    if (g >= a.R) return;
    const uint32_t grp = g * x.nsub + sub;
    const uint32_t * nmaxs = x.blk_nmax + (size_t)grp * E2_WBS;
    const uint32_t * flags = x.wbflag + (size_t)grp * E2_WBS;
    if (PASS_A) { if (nmaxs[0] == 0) return; }           // sorted: an empty first warp block means an empty group
    else {
        const int any = tid < (uint32_t)E2_WBS && flags[tid] == pass_no;
        if (!__syncthreads_or(any)) return;
    }
    if (*(volatile uint32_t *)x.ovf) return;
#ifdef PD_EM_STATS
    const long long t_blk = clock64();
#endif
    const PdRgConst * rg = a.rgc + g;
    const uint32_t hist_len = __ldg(&rg->hist_len), rows = hist_len + 1;
    const int hb = __ldg(&rg->hist_base);
    const double minp = __ldg(&rg->min_prob), lnminp = __ldg(&rg->ln_min_prob);
    // blocks with only a few warp blocks to do (late passes: a handful of pairs still iterate) read the table rows from
    // global memory instead of staging the whole table
    bool staged = true;
    if (!PASS_A) {
        const int mine = tid < (uint32_t)E2_WBS && flags[tid] == pass_no;
        staged = __syncthreads_count(mine) > 2;
    }
    const PdTab * gtab = a.tab + __ldg(&rg->hist_off);
    if (staged) {
        double2 * sA = s_tab; double * sR = reinterpret_cast<double *>(s_tab + rows), * sV = sR + rows;
        for (uint32_t r = tid; r < rows; r += E2_T) {
            const D4 v = ld4(&gtab[r].val);              // val, ln, lnp, fr
            const bool fl = v.a == minp;
            sA[r] = make_double2(v.b, fl ? v.b : v.c);
            sR[r] = fl ? -0.5 : v.d;
            sV[r] = v.a;
        }
        __syncthreads();
    }
    const uint32_t aA = (uint32_t)__cvta_generic_to_shared(s_tab), aR = aA + rows * 16u, aV = aR + rows * 8u;
    const uint32_t hl2 = hist_len - 2u;
    const uint32_t lane = tid & 31, warp = tid >> 5;
    const size_t sbase = (size_t)grp * E2_SUB;
    const double sd = __ldg(&rg->stddev);
#ifdef PD_EM_STATS
    const int so = PASS_A ? 0 : 8;
    if (tid == 0) { S2_ADD(so + 0, 1); S2_ADD(so + 1, clock64() - t_blk); }
#endif
    // the warp's warp blocks, software-pipelined: the item / control words of the next one are requested before the
    // current one is processed
    struct Pre { E2Item it; uint2 cw; E2Cur cur; uint32_t bo; };
    auto next_wb = [&](uint32_t w) -> uint32_t {          // first warp block >= w of this warp that has work
        for (; w < (uint32_t)E2_WBS; w += E2_T / 32) {
            if (nmaxs[w] == 0) return E2_WBS;
            if (PASS_A || flags[w] == pass_no) return w;
        }
        return E2_WBS;
    };
    auto fetch = [&](uint32_t w) -> Pre {
        Pre q;
        const size_t slot = sbase + w * 32 + lane;
        q.bo = x.blk_off[(size_t)grp * E2_WBS + w];
        q.it = x.item[slot];
        q.cw = *reinterpret_cast<const uint2 *>(&x.ctl[slot]);
        q.cur = E2Cur{INT_MIN, 0, 0, 0};
        if (!PASS_A) q.cur = x.cur[slot];
        return q;
    };
    uint32_t wb = next_wb(warp);
    Pre pre = Pre{E2Item{0, 0, 0, 0}, make_uint2(0, 0), E2Cur{0, 0, 0, 0}, 0};
    if (wb < (uint32_t)E2_WBS) pre = fetch(wb);
    for (; wb < (uint32_t)E2_WBS;) {
#ifdef PD_EM_STATS
        const long long t_wb = clock64();
#endif
        const uint32_t wb_cur = wb;
        const size_t slot = sbase + wb_cur * 32 + lane;
        const int4 * dp = reinterpret_cast<const int4 *>(x.devT + pre.bo) + lane;
        const E2Item it = pre.it;
        const uint2 cw = pre.cw;
        E2Cur cur = pre.cur;
        // the first read pairs of every lane are requested before the item decides whether it needs the pass
        int4 q0 = __ldg(dp), q1 = make_int4(0, 0, 0, 0);
        if (nmaxs[wb_cur] > 4) q1 = __ldg(dp + 32);
        wb = next_wb(wb_cur + E2_T / 32);
        if (wb < (uint32_t)E2_WBS) pre = fetch(wb);
        const uint32_t mode = PASS_A ? (uint32_t)E2_M2 : (cw.y >> 30);
        const int L = (int)(cw.y & E2_LMASK);
        int S = 0;
        bool need = it.n > 0;
        if (!PASS_A) {
            const int thr = hb - 1;                                            // carrier of length X: dmx >= X - hb + 1
            if (mode == E2_M1) {
                S = (int)cw.x;
                need = need && (cur.Lc == INT_MIN || S != cur.Sc || (L != cur.Lc && (it.dmx + thr >= L || it.dmx + thr >= cur.Lc)));
            } else if (mode == E2_M2) {
                need = need && (L != cur.LcA && (it.dmx + thr >= L || it.dmx + thr >= cur.LcA));
            } else need = false;
            if (mode == E2_M1 || mode == E2_M2) x.ctl[slot].lmode = cw.y & E2_LMASK;      // request consumed
        } else cur.LcA = L;
        uint32_t jmax = need ? it.n : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) jmax = max(jmax, __shfl_xor_sync(PD_FULL, jmax, o));
        if (jmax == 0) continue;
#ifdef PD_EM_STATS
        const long long t_lp = clock64();
        if (lane == 0) { S2_ADD(so + 2, 1); S2_ADD(so + 3, t_lp - t_wb); S2_ADD(so + 4, jmax); }
#endif
        const uint32_t ub = (uint32_t)(hb - 1 - S), vb = (uint32_t)(hb - 1 - L);
        const uint32_t n = need ? it.n : 0u;
        double l0 = 0, l1 = 0, l2 = 0, sr = 0, srd = 0;
        uint32_t nd = 0, c = 0; int32_t sdv = 0;
        int wlo = 0, whi = 0;
        if (PASS_A) { wlo = max(L / 2, (int)floor((double)L - 2 * sd + 0.5)); whi = (int)((double)L + 2 * sd); }
        // table in shared memory: the rows of the 4 read pairs of a load are requested together; only a read pair whose
        // deletion hypothesis lies inside the histogram (rare, and at the front of the item after k_e2_prep) takes the
        // comparing path
        auto four_s = [&](const int4 d4, const uint32_t j) {
            const int d[4] = {d4.x, d4.y, d4.z, d4.w};
            uint32_t ir[4]; bool ok[4], inr = false;
            double2 A[4]; double rbs[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                ok[k] = j + k < n;
                const uint32_t u = (uint32_t)d[k] + ub;
                ir[k] = (ok[k] && u < hl2) ? u + 2u : 0u;
                inr = inr || (ok[k] && (uint32_t)d[k] + vb < hl2);
                A[k] = lds_d2(aA + ir[k] * 16u);
                rbs[k] = lds_d(aR + ir[k] * 8u);
            }
            if (!inr) {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (ok[k]) {
                        const double r = fabs(rbs[k]);
                        nd += (uint32_t)(__double2hiint(rbs[k]) >> 31) & 1u;   // reference on the floor as well: ref == del
                        l0 += A[k].x; l1 += A[k].y; l2 += lnminp; sr += r; srd += r * d[k];
                        if (PASS_A) { c += (d[k] > wlo && d[k] < whi); sdv += d[k]; }
                    }
                return;
            }
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (ok[k]) {
                    const uint32_t v = (uint32_t)d[k] + vb;
                    double g1 = A[k].y, r = fabs(rbs[k]), ld = lnminp;
                    if (v < hl2) {                                            // deletion hypothesis inside the histogram
                        const uint32_t id = v + 2u;
                        const double ref = lds_d(aV + ir[k] * 8u), del = lds_d(aV + id * 8u);
                        const double2 dA = lds_d2(aA + id * 16u);
                        ld = dA.x;
                        if (ref == del) { g1 = A[k].x; ++nd; r = 0.5; }        // + LN2_RESIDUE in finish_triple
                        else if (del == minp) { }                              // the bulk values of the reference row
                        else if (ref == minp) { g1 = dA.y; r = 1.0 - lds_d(aR + id * 8u); }
                        else { g1 = log(ref + del) - LN2_D; r = del / (del + ref); }
                    } else nd += (uint32_t)(__double2hiint(rbs[k]) >> 31) & 1u;
                    l0 += A[k].x; l1 += g1; l2 += ld; sr += r; srd += r * d[k];
                    if (PASS_A) { c += (d[k] > wlo && d[k] < whi); sdv += d[k]; }
                }
        };
        auto one_g = [&](const int d) {                                       // table rows from global memory (pd_em.cu's dl_one)
            const uint32_t u = (uint32_t)d + ub, v = (uint32_t)d + vb;
            const uint32_t ir = u < hl2 ? u + 2u : 0u;
            const D4 rr = ld4(&gtab[ir].val);                                 // ref, ln ref, ln(ref + floor) - ln 2, floor / (floor + ref)
            double2 dv = make_double2(minp, lnminp);
            if (v < hl2) dv = ld2(&gtab[v + 2u].val);
            double g1, r;
            if (rr.a == dv.x) { g1 = rr.b; ++nd; r = 0.5; }
            else if (dv.x == minp) { g1 = rr.c; r = rr.d; }
            else if (rr.a == minp) { const double2 dq = ld2(&gtab[v + 2u].lnp); g1 = dq.x; r = 1.0 - dq.y; }
            else { g1 = log(rr.a + dv.x) - LN2_D; r = dv.x / (dv.x + rr.a); }
            l0 += rr.b; l1 += g1; l2 += dv.y; sr += r; srd += r * d;
            if (PASS_A) { c += (d > wlo && d < whi); sdv += d; }
        };
        // 4 read pairs per 128-bit load, two loads in flight while the current one is processed
        if (staged) {
            for (uint32_t j = 0; j < jmax; j += 4) {
                const int4 d = q0;
                q0 = q1;
                if (j + 8 < jmax) q1 = __ldg(dp + (size_t)((j + 8) >> 2) * 32);
                if (j < n) four_s(d, j);
            }
        } else {
            for (uint32_t j = 0; j < jmax; j += 4) {
                const int4 d = q0;
                q0 = q1;
                if (j + 8 < jmax) q1 = __ldg(dp + (size_t)((j + 8) >> 2) * 32);
                if (j < n) one_g(d.x);
                if (j + 1 < n) one_g(d.y);
                if (j + 2 < n) one_g(d.z);
                if (j + 3 < n) one_g(d.w);
            }
        }
#ifdef PD_EM_STATS
        if (lane == 0) S2_ADD(so + 5, clock64() - t_lp);
#endif
        if (need) {
            E2Rec * out = ((PASS_A || mode == E2_M2) ? x.recA : x.rec) + (size_t)it.pair * a.R + g;
            E2Rec r; r.l0 = l0; r.l1 = l1; r.l2 = l2; r.sr = sr; r.srd = srd; r.nd = nd; r.c = c; r.sd = sdv; r.pad[0] = r.pad[1] = r.pad[2] = 0;
            rec_store(out, r);
            if (!PASS_A) {
                if (mode == E2_M1) { cur.Lc = L; cur.Sc = S; } else cur.LcA = L;
                x.cur[slot] = cur;
            }
        }
    }
#ifdef PD_EM_STATS
    __syncthreads();
    if (tid == 0) S2_ADD(so + 6, clock64() - t_blk);
#endif
}

// ------------------------------------------------------------------------------------------------------------------
// pair phase
// ------------------------------------------------------------------------------------------------------------------
struct PairShared {
    double red[2][64];
    unsigned long long redu[64];
    double rgw[3];
};

struct SampleDl { double x0, E0, E1, E2; };

// likelihood triple of sample s from the records `src` of the pair
__device__ __forceinline__ SampleDl sample_dl(const PdDev & a, const uint32_t * __restrict__ cnt, const E2Rec * __restrict__ src, uint32_t s)
{
    double l0 = 0, l1 = 0, l2 = 0; uint32_t nd = 0;
    const uint32_t g0 = a.sample_rg[s], g1 = a.sample_rg[s + 1];
    for (uint32_t g = g0; g < g1; ++g) {
        const uint32_t n = cnt[g];
        if (n == 0 || n >= __ldg(&a.rgc[g].max_load)) continue;
        const E2Rec r = rec_load(src + g);
        l0 += r.l0; l1 += r.l1; l2 += r.l2; nd += r.nd;
    }
    SampleDl o; double x1, x2;
    finish_triple(l0, l1, l2, nd, o.x0, x1, x2);
    o.E0 = o.x0 == 0 ? 1.0 : exp(o.x0); o.E1 = x1 == 0 ? 1.0 : exp(x1); o.E2 = x2 == 0 ? 1.0 : exp(x2);
    return o;
}

// A pair is handled by a GROUP of threads: one warp (G = 32, cohorts of up to 128 samples: 4 samples per lane, shuffle
// reductions, no block barrier) or the whole block (G = 0).
template <int G>
struct Grp {
    __device__ static __forceinline__ uint32_t tid() { return G == 32 ? (threadIdx.x & 31u) : threadIdx.x; }
    __device__ static __forceinline__ uint32_t size() { return G == 32 ? 32u : blockDim.x; }
    __device__ static __forceinline__ void sync() { if (G == 32) __syncwarp(); else __syncthreads(); }
    __device__ static __forceinline__ void sum2(double & a, double & b, PairShared & sh, int & par)
    {
        if (G == 32) { a = warp_sum(a); b = warp_sum(b); } else block_sum2(a, b, sh.red, par);
    }
    __device__ static __forceinline__ void sum2u(unsigned long long & a, unsigned long long & b, PairShared & sh)
    {
        if (G == 32) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(PD_FULL, a, o); b += __shfl_xor_sync(PD_FULL, b, o); }
        } else block_sum2u(a, b, sh.redu);
    }
};

// one round of one pair; every exit is uniform over the group. SPT > 0: the thread's samples (tid + k * size, k < SPT)
// keep their triples in registers between the sweeps of the round; SPT = 0: they are recomputed from the records.
template <int G, int SPT>
__device__ __forceinline__ void pair_round(const PdDev & a, const EmArgs & e, const E2Args & x, PairShared & sh, const uint32_t p, const uint32_t round_no)
{
    const uint32_t tid = Grp<G>::tid(), T = Grp<G>::size();
    E2Pair & st = x.pst[p];
    const uint32_t phase = st.phase;
    if (phase >= PH_ALIVE) return;
    const PdPair pr = e.pairs[e.pair0 + p];
    const uint32_t job = pr.job - e.job_base;
    const uint32_t cj = e.cjob_of[job] - e.cj_base;
    const uint32_t * cnt = e.act_cnt + (size_t)cj * a.R;
    const E2Rec * src = (phase == PH_M1 ? x.rec : x.recA) + (size_t)p * a.R;
    const E2Rec * recA = x.recA + (size_t)p * a.R;           // sd / c of pass A
    const uint32_t * inv = x.inv + (size_t)p * a.R;
    const uint32_t nxt = (round_no + 1) % 3;
    int par = 0;
    uint32_t len = st.len, it = st.it;
    double freq = st.freq;
    Gt gt = Gt{st.gt[0], st.gt[1], st.gt[2]};
    SampleDl mine[SPT > 0 ? SPT : 1];
    if (SPT > 0) {
#pragma unroll
        for (int k = 0; k < SPT; ++k) { const uint32_t s = tid + k * T; mine[k] = SampleDl{0, 1, 1, 1}; if (s < a.N) mine[k] = sample_dl(a, cnt, src, s); }
    }
    // likelihood triple of read group 0 (rgDlIt is never advanced, :401,424-431: it drives every reference shift)
    double r0 = 0, r1 = 0, r2 = 0;
    if (tid == T - 1) {
        const uint32_t n0 = cnt[0];
        if (n0 < __ldg(&a.rgc[0].max_load)) {             // else Triple(0,0,0) like the reference
            double l0 = 0, l1 = 0, l2 = 0;
            if (n0) { const E2Rec r = rec_load(src); l0 = r.l0; l1 = r.l1; l2 = r.l2; }
            const double m = fmax(fmax(l0, l1), l2);
            r0 = exp(l0 - m); r1 = exp(l1 - m); r2 = exp(l2 - m);
        }
        if (G != 32) { sh.rgw[0] = r0; sh.rgw[1] = r1; sh.rgw[2] = r2; }
    }
    if (G == 32) { r0 = __shfl_sync(PD_FULL, r0, 31); r1 = __shfl_sync(PD_FULL, r1, 31); r2 = __shfl_sync(PD_FULL, r2, 31); }
    else { __syncthreads(); r0 = sh.rgw[0]; r1 = sh.rgw[1]; r2 = sh.rgw[2]; }
    // f(sample index, its triple) for every sample of this thread
    auto for_samples = [&](auto f) {
        if (SPT > 0) {
#pragma unroll
            for (int k = 0; k < SPT; ++k) { const uint32_t s = tid + k * T; if (s < a.N) f(s, mine[k]); }
        } else {
            for (uint32_t s = tid; s < a.N; s += T) f(s, sample_dl(a, cnt, src, s));
        }
    };
    auto lr_now = [&](const Gt g) {                      // deletion_likelihood_ratio :490-508
        double del = 0, nodel = 0;
        for_samples([&](uint32_t, const SampleDl & d) {
            const double p0 = d.E0 * g.a, p1 = d.E1 * g.b, p2 = d.E2 * g.c, pAll = p0 + p1 + p2;
            del += log(p0 / pAll * d.E0 + p1 / pAll * d.E1 + p2 / pAll * d.E2);
            nodel += d.x0;
        });
        Grp<G>::sum2(del, nodel, sh, par);
        return del - nodel;
    };
    auto request = [&](uint32_t lm) {                    // next pass for every item of the pair
        for (uint32_t g = tid; g < a.R; g += T) {
            const uint32_t q = inv[g];
            x.ctl[q].lmode = lm;
            x.wbflag[q >> 5] = round_no + 1;
        }
        if (tid == 0) x.act[(size_t)nxt * x.npairs + atomicAdd(x.actn + nxt, 1u)] = p;
    };
    auto finish = [&](bool alive, uint32_t src_a, uint32_t reason) {
        // request the final pass (alive) or publish the rejection
        if (alive) {
            for (uint32_t s = tid; s < a.N; s += T) {
                const uint32_t g0 = a.sample_rg[s], g1 = a.sample_rg[s + 1];
                int lo = INT_MAX, hi = 0;                // borders of the LAST usable read group apply to the whole sample (quirk)
                for (uint32_t g = g0; g < g1; ++g) {
                    if (cnt[g] >= __ldg(&a.rgc[g].max_load)) continue;
                    lo = (int)len - __ldg(&a.rgc[g].lower_q); hi = (int)len + __ldg(&a.rgc[g].upper_q);
                }
                for (uint32_t g = g0; g < g1; ++g) {
                    const uint32_t q = inv[g];
                    E2Ctl * c = x.ctl + q;
                    if (src_a) c->shift = 0;
                    c->supp_lo = lo; c->supp_hi = hi;
                    c->lmode = (len & E2_LMASK) | ((uint32_t)E2_FIN << 30);
                    x.finflag[q >> 5] = 1;
                }
            }
        }
        if (tid == 0) {
            st.len = len; st.it = it; st.freq = freq; st.gt[0] = gt.a; st.gt[1] = gt.b; st.gt[2] = gt.c;
            st.src_a = src_a; st.phase = alive ? PH_ALIVE : PH_DEAD;
            if (alive) x.alive[atomicAdd(x.actn + 3, 1u)] = p;
            else {
                e.valid[p] = 0;
                if (e.dbg) { e.dbg[4 * p] = reason; e.dbg[4 * p + 1] = len; e.dbg[4 * p + 2] = it; }
                __threadfence();
                st_release_gpu(e.done + p, 1u);
            }
        }
    };

    if (phase == PH_A) {
        // ---- initialize_allele_frequency :93-133
        unsigned long long c = 0, t = 0;
        for (uint32_t s = tid; s < a.N; s += T)
            for (uint32_t g = a.sample_rg[s]; g < a.sample_rg[s + 1]; ++g) {
                const uint32_t n = cnt[g];
                if (n == 0 || n >= __ldg(&a.rgc[g].max_load)) continue;
                t += n; c += recA[g].c;
            }
        Grp<G>::sum2u(c, t, sh);
        freq = t == 0 ? 0.0 : (double)c / (double)t;
        gt = gt_prior(freq, e.somatic);
        if (freq == 0) { finish(false, 0, 1); return; }
    } else if (phase == PH_M1) {
        // ---- update_allele_frequency :467-485 (priors of the previous iteration)
        double fs = 0, dummy = 0;
        for_samples([&](uint32_t, const SampleDl & d) {
            const double p0 = d.E0 * gt.a, p1 = d.E1 * gt.b, p2 = d.E2 * gt.c;
            fs += (p1 + 2 * p2) / (p0 + p1 + p2);
        });
        Grp<G>::sum2(fs, dummy, sh, par);
        freq = fs / 2.0 / a.N;
        if (freq == 0) { finish(false, 0, 2); return; }
        gt = gt_prior(freq, e.somatic);
        bool conv = false;
        for (uint32_t i = 0; i < st.nvisited; ++i)
            if (st.vlen[i] == (int)len && fabs(st.vfreq[i] - freq) <= 0.0001) conv = true;
        if (conv) {
            // convergence :632-658: compare with the previous estimate evaluated with the initial (zero) shifts
            const double lr = lr_now(gt);
            request((st.prev_len & E2_LMASK) | ((uint32_t)E2_M2 << 30));
            if (tid == 0) {
                st.lr_conv = lr; st.freq = freq; st.gt[0] = gt.a; st.gt[1] = gt.b; st.gt[2] = gt.c; st.phase = PH_M2;
            }
            return;
        }
    } else {                                             // PH_M2: the records in recA hold the previous estimate
        const double plr = lr_now(gt_prior(st.prev_freq, e.somatic));
        uint32_t src_a = 0;
        if (plr > st.lr_conv) { len = st.prev_len; freq = st.prev_freq; src_a = 1; }
        const bool alive = !(freq < 0.0000000001 || len < e.min_len);
        finish(alive, src_a, 2);
        return;
    }
    if (!(len >= e.min_len && it < e.iterations)) {
        const bool alive = !(freq < 0.0000000001 || len < e.min_len);
        finish(alive, phase == PH_A ? 1u : 0u, 2);           // without an iteration the records of pass A are the final state
        return;
    }
    // ---- next iteration: update_deletion_length :388-462 from the moments of the posterior weights
    ++it;
    const uint32_t prevLen = len; const double prevFreq = freq;
    const double aSumRg = r0 * gt.a + r1 * gt.b + r2 * gt.c;
    const double ea0Rg = r0 * gt.a / aSumRg, ea1Rg = r1 * gt.b / aSumRg;          // NaN when read group 0 is high-coverage
    double sumDel = 0, wDel = 0;
    const bool single = a.R == a.N;                      // one read group per sample: the shifts stay in registers until the new
    int my_sft[SPT > 0 ? SPT : 1];                       // length is known and go out with it in one 8-byte store per item
    int kk = 0;
    for_samples([&](uint32_t s, const SampleDl & d) {
        const double invp = 1.0 / (d.E0 * gt.a + d.E1 * gt.b + d.E2 * gt.c);
        const double ea1 = d.E1 * gt.b * invp, ea2 = d.E2 * gt.c * invp;
        for (uint32_t g = a.sample_rg[s]; g < a.sample_rg[s + 1]; ++g) {
            const uint32_t n = cnt[g];
            if (n >= __ldg(&a.rgc[g].max_load)) { if (SPT > 0 && single) my_sft[kk] = 0; continue; }
            double Sr = 0, Srd = 0, Sd = 0; const double dn = (double)n;
            if (n) { const E2Rec r = rec_load(src + g); Sr = r.sr; Srd = r.srd; Sd = (double)(phase == PH_A ? r.sd : recA[g].sd); }
            sumDel += ea1 * Sr + ea2 * dn; wDel += ea1 * Srd + ea2 * Sd;
            const double sumRef = ea1Rg * (dn - Sr) + ea0Rg * dn, wRef = ea1Rg * (Sd - Srd) + ea0Rg * Sd;
            const double q = wRef / sumRef;
            int sft = (q != q) ? 0 : (q >= 2147483647.0 ? INT_MAX : (q <= -2147483648.0 ? INT_MIN : (int)q));
            const double sdg = __ldg(&a.rgc[g].stddev);
            if (sft > sdg || sft < -1 * sdg) sft = 0;
            if (SPT > 0 && single) my_sft[kk] = sft; else x.ctl[inv[g]].shift = sft;
        }
        ++kk;
    });
    Grp<G>::sum2(sumDel, wDel, sh, par);
    if (sumDel == 0) len = 0;
    else { const double nlen = wDel / sumDel; len = nlen < 0 ? 0u : (uint32_t)round(nlen); }
    if (SPT > 0 && single) {
        const uint32_t lm = (len & E2_LMASK) | ((uint32_t)E2_M1 << 30);
#pragma unroll
        for (int k = 0; k < (SPT > 0 ? SPT : 1); ++k) {
            const uint32_t g = tid + k * T;
            if (g < a.R) {
                const uint32_t q = inv[g];
                *reinterpret_cast<uint2 *>(&x.ctl[q]) = make_uint2((uint32_t)my_sft[k], lm);
                x.wbflag[q >> 5] = round_no + 1;
            }
        }
        if (tid == 0) x.act[(size_t)nxt * x.npairs + atomicAdd(x.actn + nxt, 1u)] = p;
    } else request((len & E2_LMASK) | ((uint32_t)E2_M1 << 30));
    if (tid == 0) {
        int f = -1;                                      // visited[prevLen] = prevFreq (:600)
        const int nv = (int)st.nvisited;
        for (int i = 0; i < nv; ++i) if (st.vlen[i] == (int)prevLen) f = i;
        if (f < 0) { f = nv; st.vlen[f] = (int)prevLen; st.nvisited = (uint32_t)nv + 1; }
        st.vfreq[f] = prevFreq;
        st.len = len; st.it = it; st.prev_len = prevLen; st.freq = freq; st.prev_freq = prevFreq;
        st.gt[0] = gt.a; st.gt[1] = gt.b; st.gt[2] = gt.c; st.phase = PH_M1;
    }
}

// persistent groups over the list of pairs that asked for the pass that has just run (round 0: every pair)
template <int TPB, int G, int SPT>
__global__ void __launch_bounds__(TPB) k_e2_pair(PdDev a, EmArgs e, E2Args x, uint32_t round_no)
{
    __shared__ PairShared sh;
    if (*(volatile uint32_t *)x.ovf) return;
    const uint32_t cur = round_no % 3;
    const uint32_t count = round_no == 0 ? x.npairs : x.actn[cur];
    if (blockIdx.x == 0 && threadIdx.x == 0) x.actn[(round_no + 2) % 3] = 0;          // the list after the next one
    const uint32_t gpb = G == 32 ? TPB / 32 : 1;          // groups per block
    const uint32_t gid = blockIdx.x * gpb + (G == 32 ? threadIdx.x >> 5 : 0);
    for (uint32_t i = gid; i < count; i += gridDim.x * gpb) {
        const uint32_t p = round_no == 0 ? i : x.act[(size_t)cur * x.npairs + i];
        Grp<G>::sync();
        pair_round<G, SPT>(a, e, x, sh, p, round_no);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// final pass
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(E2_T, 4) k_e2_final_reads(PdDev a, EmArgs e, E2Args x)
{
    extern __shared__ double2 s_tab[];                   // [rows] {log10, log10p}, then [rows] val (double)
    const uint32_t tid = threadIdx.x, sub = blockIdx.x, g = pd_grid_row();
    if (g >= a.R) return;
    const uint32_t grp = g * x.nsub + sub;
    const uint32_t * nmaxs = x.blk_nmax + (size_t)grp * E2_WBS;
    const uint32_t * flags = x.finflag + (size_t)grp * E2_WBS;
    {
        const int any = tid < (uint32_t)E2_WBS && flags[tid] != 0 && nmaxs[tid] != 0;
        if (!__syncthreads_or(any)) return;
    }
    if (*(volatile uint32_t *)x.ovf) return;
    const PdRgConst * rg = a.rgc + g;
    const uint32_t hist_len = __ldg(&rg->hist_len), rows = hist_len + 1;
    const int hb = __ldg(&rg->hist_base);
    const double minp = __ldg(&rg->min_prob), l10minp = __ldg(&rg->l10_min_prob);
    const int lower_q = __ldg(&rg->lower_q), upper_q = __ldg(&rg->upper_q), inner_off = __ldg(&rg->inner_off);
    const uint32_t lane = tid & 31, warp = tid >> 5;
    const size_t sbase = (size_t)grp * E2_SUB;
    double2 * sC = s_tab; double * sV = reinterpret_cast<double *>(s_tab + rows);
    {
        const PdTab * t = a.tab + __ldg(&rg->hist_off);
        for (uint32_t r = tid; r < rows; r += E2_T) {
            sC[r] = ld2(&t[r].l10);
            sV[r] = __ldg(&t[r].val);
        }
    }
    __syncthreads();
    const uint32_t hl2 = hist_len - 2u;
    for (uint32_t wb = warp; wb < (uint32_t)E2_WBS; wb += E2_T / 32) {
        if (nmaxs[wb] == 0) break;
        if (flags[wb] == 0) continue;
        const size_t slot = sbase + wb * 32 + lane;
        const E2Item it = x.item[slot];
        const E2Ctl cw = x.ctl[slot];
        const bool need = (cw.lmode >> 30) == E2_FIN && it.n > 0;
        uint32_t jmax = need ? it.n : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) jmax = max(jmax, __shfl_xor_sync(PD_FULL, jmax, o));
        if (jmax == 0) continue;
        const int flen = (int)(cw.lmode & E2_LMASK);
        const size_t bo = (size_t)x.blk_off[(size_t)grp * E2_WBS + wb];
        const int4 * dp = reinterpret_cast<const int4 *>(x.devT + bo) + lane;
        const uint4 * pp = reinterpret_cast<const uint4 *>(x.posT + bo) + lane;
        const uint32_t ub = (uint32_t)(hb - 1 - cw.shift), vb = (uint32_t)(hb - 1 - flen);
        const uint32_t n = need ? it.n : 0u;
        const int delLower = flen - lower_q, delUpper = flen + upper_q;           // DAD: the read group's own borders
        double t0 = 0, t1 = 0, t2 = 0;
        uint32_t lad0 = 0, lad1 = 0, lad2 = 0, dad0 = 0, dad1 = 0, dad2 = 0, dad3 = 0, dad4 = 0, fl_min = 0xFFFFFFFFu, fl_max = 0, nsupp = 0;
        auto one = [&](const int d, const uint32_t pos) {
            if (d > upper_q) { if (d < delLower) ++dad2; else if (d <= delUpper) ++dad3; else ++dad4; }
            else { if (d < delUpper) ++dad0; else ++dad1; }
            const uint32_t u = (uint32_t)d + ub, v = (uint32_t)d + vb;
            const uint32_t ir = u < hl2 ? u + 2u : 0u;
            const double2 rc = sC[ir]; const double ref = sV[ir];
            double del = minp; double2 dc = make_double2(l10minp, 0.0);
            if (v < hl2) { dc = sC[v + 2u]; del = sV[v + 2u]; }
            if (ref >= 2 * del) ++lad0; else if (del >= 2 * ref) ++lad2; else ++lad1;
            t0 += rc.x; t2 += dc.x;
            if (ref == del) t1 += rc.x;                                       // residue applied in k_e2_final_pair
            else if (del == minp) t1 += rc.y;
            else if (ref == minp) t1 += dc.y;
            else t1 += log10(ref + del) - LOG10_2_D;
            const uint32_t first = pos + e.anchor;
            const uint32_t last = first + (uint32_t)max(0, d + inner_off);
            fl_min = min(fl_min, first); fl_max = max(fl_max, last);
            nsupp += (d >= cw.supp_lo && d <= cw.supp_hi);                    // supporting read pair
        };
        int4 nd4 = make_int4(0, 0, 0, 0); uint4 np4 = make_uint4(0, 0, 0, 0);
        if (n) { nd4 = __ldg(dp); np4 = __ldg(pp); }
        for (uint32_t j = 0; j < jmax; j += 4) {
            const int4 d = nd4; const uint4 q = np4;
            if (j + 4 < n) { nd4 = __ldg(dp + (size_t)((j + 4) >> 2) * 32); np4 = __ldg(pp + (size_t)((j + 4) >> 2) * 32); }
            if (j < n) one(d.x, q.x);
            if (j + 1 < n) one(d.y, q.y);
            if (j + 2 < n) one(d.z, q.z);
            if (j + 3 < n) one(d.w, q.w);
        }
        if (need) {
            E2Fin f;
            f.t0 = t0; f.t1 = t1; f.t2 = t2; f.lad[0] = lad0; f.lad[1] = lad1; f.lad[2] = lad2;
            f.dad[0] = dad0; f.dad[1] = dad1; f.dad[2] = dad2; f.dad[3] = dad3; f.dad[4] = dad4;
            f.fl_min = fl_min; f.fl_max = fl_max; f.nsupp = nsupp; f.pad[0] = f.pad[1] = f.pad[2] = 0;
            rec_store(x.fin + (size_t)it.pair * a.R + g, f);
            if (nsupp) {                                                      // second walk: append the supporting read pairs
                uint32_t k = atomicAdd(x.suppn + it.pair, nsupp);
                uint32_t * of = x.supp_first + (size_t)it.pair * E2_SUPP_CAP, * ol = x.supp_last + (size_t)it.pair * E2_SUPP_CAP;
                const int32_t * d1 = x.devT + bo + lane * 4; const uint32_t * p1 = x.posT + bo + lane * 4;
                for (uint32_t j = 0; j < n; ++j) {
                    const size_t o = (size_t)(j >> 2) * 128 + (j & 3);
                    const int d = d1[o];
                    if (d >= cw.supp_lo && d <= cw.supp_hi) {
                        if (k < E2_SUPP_CAP) { const uint32_t first = p1[o] + e.anchor; of[k] = first; ol[k] = first + (uint32_t)max(0, d + inner_off); }
                        ++k;
                    }
                }
            }
        }
    }
}

template <int TPB>
__global__ void __launch_bounds__(TPB) k_e2_final_pair(PdDev a, EmArgs e, E2Args x)
{
    __shared__ PairShared sh;
    __shared__ uint32_t s_first[E2_SUPP_CAP], s_last[E2_SUPP_CAP];
    __shared__ uint32_t s_sel[2];
    if (*(volatile uint32_t *)x.ovf) return;
    const uint32_t tid = threadIdx.x, T = blockDim.x;
    const uint32_t count = x.actn[3];
    for (uint32_t ai = blockIdx.x; ai < count; ai += gridDim.x) {
    const uint32_t p = x.alive[ai];
    __syncthreads();
    E2Pair & st = x.pst[p];
    const PdPair pr = e.pairs[e.pair0 + p];
    const uint32_t job = pr.job - e.job_base;
    const uint32_t w = e.job_window[pr.job];
    const uint32_t cj = e.cjob_of[job] - e.cj_base;
    const uint32_t * cnt = e.act_cnt + (size_t)cj * a.R;
    const uint32_t * off = e.act_off + (size_t)cj * a.R;
    const E2Rec * src = (st.src_a ? x.recA : x.rec) + (size_t)p * a.R;
    const E2Fin * fin = x.fin + (size_t)p * a.R;
    const uint8_t * sstat = e.sstat + (size_t)job * a.N;
    uint32_t * ps = e.ps + (size_t)p * 13 * a.N;
    const int len = (int)st.len;
    const Gt gt = Gt{st.gt[0], st.gt[1], st.gt[2]};
    int par = 0;
    auto reject = [&](uint32_t reason) {
        if (tid == 0) {
            e.valid[p] = 0; st.phase = PH_DONE;
            if (e.dbg) { e.dbg[4 * p] = reason; e.dbg[4 * p + 1] = st.len; e.dbg[4 * p + 2] = st.it; }
            __threadfence();
            st_release_gpu(e.done + p, 1u);
        }
    };
    unsigned long long supp = 0, ndata = 0;
    double del = 0, nodel = 0;
    for (uint32_t s = tid; s < a.N; s += T) {
        uint32_t lad0 = 0, lad1 = 0, lad2 = 0, dad0 = 0, dad1 = 0, dad2 = 0, dad3 = 0, dad4 = 0, fl_min = 0xFFFFFFFFu, fl_max = 0, ndeg = 0;
        double l0 = 0, l1 = 0, l2 = 0, t0 = 0, t1 = 0, t2 = 0;
        for (uint32_t g = a.sample_rg[s]; g < a.sample_rg[s + 1]; ++g) {
            const uint32_t n = cnt[g];
            if (n == 0 || n >= __ldg(&a.rgc[g].max_load)) continue;
            const E2Rec r = rec_load(src + g); const E2Fin f = rec_load(fin + g);
            l0 += r.l0; l1 += r.l1; l2 += r.l2; ndeg += r.nd;
            t0 += f.t0; t1 += f.t1; t2 += f.t2;
            lad0 += f.lad[0]; lad1 += f.lad[1]; lad2 += f.lad[2];
            dad0 += f.dad[0]; dad1 += f.dad[1]; dad2 += f.dad[2]; dad3 += f.dad[3]; dad4 += f.dad[4];
            fl_min = min(fl_min, f.fl_min); fl_max = max(fl_max, f.fl_max);
            supp += f.nsupp;
        }
        if (fl_min == 0xFFFFFFFFu) fl_min = 0;
        double x0, x1, x2, g0l = t0, g1l = t1, g2l = t2;
        if (t0 + t1 + t2 == 0.0) { x0 = 0; x1 = LN1E10; x2 = LN1E10; }       // sum(gtLogs) == 0 :307-308
        else {
            const double mg = fmax(fmax(t0, t1), t2);
            g0l -= mg; g1l -= mg; g2l -= mg;
            if (ndeg) { g1l += ndeg * LOG10_2_RESIDUE; const double m2 = fmax(fmax(g0l, g1l), g2l); g0l -= m2; g1l -= m2; g2l -= m2; }
            if (g0l == g1l && g0l == g2l) { g0l = 0; g1l = -10; g2l = -10; }
            finish_triple(l0, l1, l2, ndeg, x0, x1, x2);
        }
        const double E0 = exp(x0), E1 = exp(x1), E2 = exp(x2);
        // calculatePhredGL utils_popdel.h:1511-1528
        const double gTot = log10(exp(g0l) + exp(g1l) + exp(g2l));
        const double q0 = -10 * (g0l - gTot), q1 = -10 * (g1l - gTot), q2 = -10 * (g2l - gTot);
        const double mn = fmin(fmin(q0, q1), q2);
        uint32_t * o = ps + 13 * s;
        const bool low = sstat[s] == 0;
        o[0] = low ? 0u : (uint32_t)round(q0 - mn);
        o[1] = low ? 0u : (uint32_t)round(q1 - mn);
        o[2] = low ? 0u : (uint32_t)round(q2 - mn);
        o[3] = lad0; o[4] = lad1; o[5] = lad2;
        o[6] = dad0; o[7] = dad1; o[8] = dad2; o[9] = dad3; o[10] = dad4;
        o[11] = fl_min; o[12] = fl_max;
        if (!low) ++ndata;
        // deletion_likelihood_ratio :490-508
        const double p0 = E0 * gt.a, p1 = E1 * gt.b, p2 = E2 * gt.c, pAll = p0 + p1 + p2;
        del += log(p0 / pAll * E0 + p1 / pAll * E1 + p2 / pAll * E2);
        nodel += x0;
    }
    block_sum2u(supp, ndata, sh.redu);
    if (supp == 0) { reject(3); continue; }
    // percentiles of the supporting starts (80th) and ends (20th): getSuppFirstLast :514-529, by value bisection
    const unsigned long long kF = (unsigned long long)round((double)(supp - 1) * 0.8);
    const unsigned long long kL = (unsigned long long)round((double)(supp - 1) * (1 - 0.8));
    uint32_t sF, sL;
    if (supp <= E2_SUPP_CAP) {
        const uint32_t ns = (uint32_t)supp;
        for (uint32_t i = tid; i < ns; i += T) { s_first[i] = x.supp_first[(size_t)p * E2_SUPP_CAP + i]; s_last[i] = x.supp_last[(size_t)p * E2_SUPP_CAP + i]; }
        __syncthreads();
        if (tid < 32) {
            uint32_t loF = 0xFFFFFFFFu, hiF = 0, loL = 0xFFFFFFFFu, hiL = 0;
            for (uint32_t i = tid; i < ns; i += 32) { loF = min(loF, s_first[i]); hiF = max(hiF, s_first[i]); loL = min(loL, s_last[i]); hiL = max(hiL, s_last[i]); }
            for (int o = 16; o > 0; o >>= 1) {
                loF = min(loF, __shfl_xor_sync(PD_FULL, loF, o)); hiF = max(hiF, __shfl_xor_sync(PD_FULL, hiF, o));
                loL = min(loL, __shfl_xor_sync(PD_FULL, loL, o)); hiL = max(hiL, __shfl_xor_sync(PD_FULL, hiL, o));
            }
            while (loF < hiF || loL < hiL) {
                const uint32_t midF = loF + (hiF - loF) / 2, midL = loL + (hiL - loL) / 2;
                uint32_t cF = 0, cL = 0;
                for (uint32_t i = tid; i < ns; i += 32) { cF += s_first[i] <= midF; cL += s_last[i] <= midL; }
                for (int o = 16; o > 0; o >>= 1) { cF += __shfl_xor_sync(PD_FULL, cF, o); cL += __shfl_xor_sync(PD_FULL, cL, o); }
                if (loF < hiF) { if (cF >= kF + 1) hiF = midF; else loF = midF + 1; }
                if (loL < hiL) { if (cL >= kL + 1) hiL = midL; else loL = midL + 1; }
            }
            if (tid == 0) { s_sel[0] = loF; s_sel[1] = loL; }
        }
        __syncthreads();
        sF = s_sel[0]; sL = s_sel[1];
    } else {
        // more supporting read pairs than the list holds: bisect on the value, recounting from the pool each step
        uint32_t loF = 0, hiF = 0xFFFFFFFFu, loL = 0, hiL = 0xFFFFFFFFu;
        while (loF < hiF || loL < hiL) {
            const uint32_t midF = loF + (hiF - loF) / 2, midL = loL + (hiL - loL) / 2;
            unsigned long long cF = 0, cL = 0;
            for (uint32_t s = tid; s < a.N; s += T) {
                int delLower = INT_MAX, delUpper = 0;
                const uint32_t g0 = a.sample_rg[s], g1 = a.sample_rg[s + 1];
                for (uint32_t g = g0; g < g1; ++g) {
                    if (cnt[g] >= __ldg(&a.rgc[g].max_load)) continue;
                    delLower = len - __ldg(&a.rgc[g].lower_q); delUpper = len + __ldg(&a.rgc[g].upper_q);
                }
                for (uint32_t g = g0; g < g1; ++g) {
                    const uint32_t n = cnt[g];
                    if (n >= __ldg(&a.rgc[g].max_load)) continue;
                    const int inner_off = __ldg(&a.rgc[g].inner_off);
                    const uint32_t * pp = e.pool_pos + off[g];
                    const int32_t * pd = e.pool_dev + off[g];
                    for (uint32_t i = 0; i < n; ++i) {
                        const int d = pd[i];
                        if (d >= delLower && d <= delUpper) {
                            const uint32_t first = pp[i] + e.anchor;
                            const uint32_t last = first + (uint32_t)max(0, d + inner_off);
                            cF += first <= midF; cL += last <= midL;
                        }
                    }
                }
            }
            block_sum2u(cF, cL, sh.redu);
            if (loF < hiF) { if (cF >= kF + 1) hiF = midF; else loF = midF + 1; }
            if (loL < hiL) { if (cL >= kL + 1) hiL = midL; else loL = midL + 1; }
        }
        sF = loF; sL = loL;
    }
    if (sF == 0 && sL == 0) { reject(4); continue; }
    block_sum2(del, nodel, sh.red, par);
    const double lr = del - nodel;
    if (tid == 0) {
        const bool ok = lr >= e.min_lr;
        e.valid[p] = ok ? 1 : 0;
        st.phase = PH_DONE;
        if (e.dbg) { e.dbg[4 * p] = ok ? 0 : 5; e.dbg[4 * p + 1] = st.len; e.dbg[4 * p + 2] = st.it; e.dbg[4 * p + 3] = (uint32_t)supp; }
        if (ok) {
            pd_call c;
            c.initial_length = (uint32_t)pr.L0; c.iterations = st.it; c.deletion_length = st.len;
            c.filter = ((double)ndata / a.N >= e.min_sample_fraction) ? 0u : 4u;
            c.lr = lr; c.frequency = st.freq;
            const uint32_t cur = e.anchor + w * PD_WIN;
            c.window_position = cur - 1;
            c.position = e.window_wise ? cur - 1 : sF;
            c.end_position = e.window_wise ? 0u : sL;
            c.segment = (uint32_t)(((uint64_t)w * PD_WIN) / a.window_buffer);
            e.calls[p] = c;
        }
        __threadfence();
        st_release_gpu(e.done + p, 1u);
    }
    }
}

template <typename T>
int e2_grow(pd_ctx * c, int slot, T *& p, size_t count)
{
    void * q = nullptr;
    if (pd_grow_scratch(c, slot, std::max<size_t>(count, 1) * sizeof(T), &q)) return c->status;
    p = reinterpret_cast<T *>(q);
    return 0;
}

}  // namespace

// bytes of scratch one pair needs in the pipeline above (sizes the EM chunks in pd_scan.cu)
size_t pd_em2_pair_bytes(uint32_t R, double reads_per_pair)
{
    return (size_t)R * (3 * 16 + 2 * 64 + 4 + 80 + 8) + sizeof(E2Pair) + (size_t)E2_SUPP_CAP * 8 + (size_t)(reads_per_pair * 8 * 1.3) + 64;
}

bool pd_em2_usable(const pd_ctx * c)
{
    if (getenv("PD_EM_V1") || getenv("PD_EM_GENERAL")) return false;
    uint32_t rows = 0;
    for (const auto & k : c->rgc) rows = std::max(rows, k.hist_len + 1);
    if ((size_t)rows * 32 > 160 * 1024) return false;
    // Measured on B200 (profiles/r02): cohorts of up to 256 single-read-group samples are still faster through the fused
    // pair-major kernel (k_em_one: 2.25 vs 2.47 ms per chr21 step at 100 samples); everything else -- several read
    // groups per sample, larger cohorts (10 000 samples x 1 Mbp: 8.0 vs 22.9 ms) -- goes through this pipeline.
    // PD_EM_V2=1 forces it (tests).
    if (getenv("PD_EM_V2")) return true;
    return !(c->R == c->N && c->N <= 256);
}

int pd_launch_em2(pd_ctx * c, const PdDev & a, const EmArgs & e, double reads_per_pair, cudaStream_t st, uint64_t * launches)
{
    const uint32_t np = e.npairs, R = a.R, N = a.N;
    if (np == 0) return 0;
    E2Args x;
    x.nsub = (np + E2_SUB - 1) / E2_SUB; x.npairs = np;
    const size_t groups = (size_t)R * x.nsub, slots = groups * E2_SUB, items = (size_t)np * R;
    uint32_t * flags2;
    if (e2_grow(c, PD_S_E2_ITEM, x.item, slots) || e2_grow(c, PD_S_E2_CTL, x.ctl, slots) || e2_grow(c, PD_S_E2_CUR, x.cur, slots) ||
        e2_grow(c, PD_S_E2_REC, x.rec, items) || e2_grow(c, PD_S_E2_RECA, x.recA, items) ||
        e2_grow(c, PD_S_E2_INV, x.inv, items) || e2_grow(c, PD_S_E2_FIN, x.fin, items) || e2_grow(c, PD_S_E2_PST, x.pst, (size_t)np) ||
        e2_grow(c, PD_S_E2_BOFF, x.blk_off, groups * E2_WBS) || e2_grow(c, PD_S_E2_BNMAX, x.blk_nmax, groups * E2_WBS) ||
        e2_grow(c, PD_S_E2_FLAGS, flags2, 2 * groups * E2_WBS) || e2_grow(c, PD_S_E2_ACT, x.act, (size_t)4 * np) ||
        e2_grow(c, PD_S_E2_SUPPN, x.suppn, (size_t)np + 8) || e2_grow(c, PD_S_E2_SUPPF, x.supp_first, (size_t)np * E2_SUPP_CAP) ||
        e2_grow(c, PD_S_E2_SUPPL, x.supp_last, (size_t)np * E2_SUPP_CAP))
        return c->status;
    x.wbflag = flags2; x.finflag = flags2 + groups * E2_WBS;
    x.alive = x.act + (size_t)3 * np;
    // lane-interleaved read-pair copies: capacity from the pool density of this batch, kept across scans; k_e2_prep reports
    // an overflow and the scan is repeated with the exact need (pd_scan.cu)
    const size_t want = (size_t)(reads_per_pair * np * 1.3) + groups * 4096 + (1u << 20);
    if (want > c->e2_devt_cap) c->e2_devt_cap = want;
    if (c->e2_devt_cap > 0xFFFFFF00ull) c->e2_devt_cap = 0xFFFFFF00ull;
    if (e2_grow(c, PD_S_E2_DEVT, x.devT, c->e2_devt_cap) || e2_grow(c, PD_S_E2_POST, x.posT, c->e2_devt_cap)) return c->status;
    x.devt_cap = (uint32_t)c->e2_devt_cap;
    uint32_t * cnts;
    if (e2_grow(c, PD_S_E2_CNT, cnts, (size_t)8)) return c->status;
    x.devt_used = cnts; x.ovf = cnts + 1; x.actn = cnts + 2;                // [2..5]: list counts; ovf is sticky for the scan (cleared by pd_run_scan)
    PD_CUDA(c, cudaMemsetAsync(x.devt_used, 0, 4, st));
    PD_CUDA(c, cudaMemsetAsync(x.actn, 0, 16, st));
    PD_CUDA(c, cudaMemsetAsync(x.suppn, 0, (size_t)np * 4, st));

    uint32_t rows = 0;
    for (const auto & k : c->rgc) rows = std::max(rows, k.hist_len + 1);
    const size_t smem_em = (size_t)rows * 32, smem_fin = (size_t)rows * 24;
    if (smem_em > 48 * 1024) {
        PD_CUDA(c, cudaFuncSetAttribute(k_e2_reads<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_em));
        PD_CUDA(c, cudaFuncSetAttribute(k_e2_reads<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_em));
    }
    if (smem_fin > 48 * 1024) PD_CUDA(c, cudaFuncSetAttribute(k_e2_final_reads, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_fin));
    const dim3 gg = pd_rows_grid(x.nsub, R);
    // pair phase: one warp per pair for cohorts of up to 128 samples, else one block per pair
    const uint32_t TP = N <= 128 ? 256 : (N <= 256 ? 256 : (N <= 512 ? 512 : 1024));
    const uint32_t gpb = N <= 128 ? 8 : 1;
    const uint32_t pgrid_full = std::min<uint32_t>((np + gpb - 1) / gpb, 148u * (2048u / TP));
    auto pair = [&](uint32_t round_no) {
        // after the first rounds only a few pairs still iterate: a small grid keeps the fixed cost of the round low
        const uint32_t pgrid = round_no < 5 ? pgrid_full : std::min<uint32_t>(pgrid_full, 148u);
        if (N <= 128) k_e2_pair<256, 32, 4><<<pgrid, 256, 0, st>>>(a, e, x, round_no);
        else if (N <= 256) k_e2_pair<256, 0, 1><<<pgrid, 256, 0, st>>>(a, e, x, round_no);
        else if (N <= 512) k_e2_pair<512, 0, 1><<<pgrid, 512, 0, st>>>(a, e, x, round_no);
        else if (N <= 1024) k_e2_pair<1024, 0, 1><<<pgrid, 1024, 0, st>>>(a, e, x, round_no);
        else k_e2_pair<1024, 0, 0><<<pgrid, 1024, 0, st>>>(a, e, x, round_no);
    };
    const uint32_t TF = N <= 128 ? 128 : TP;
    const uint32_t fgrid = std::min<uint32_t>(np, 148u * (2048u / TF));
    k_e2_prep<<<gg, E2_T, 0, st>>>(a, e, x);
    k_e2_reads<true><<<gg, E2_T, smem_em, st>>>(a, e, x, 0u);
    pair(0);
    *launches += 3;
    for (uint32_t r = 0; r < e.iterations + 1; ++r) {
        k_e2_reads<false><<<gg, E2_T, smem_em, st>>>(a, e, x, r + 1);
        pair(r + 1);
        *launches += 2;
    }
    k_e2_final_reads<<<gg, E2_T, smem_fin, st>>>(a, e, x);
    if (TF == 128) k_e2_final_pair<128><<<fgrid, 128, 0, st>>>(a, e, x);
    else if (TF == 256) k_e2_final_pair<256><<<fgrid, 256, 0, st>>>(a, e, x);
    else if (TF == 512) k_e2_final_pair<512><<<fgrid, 512, 0, st>>>(a, e, x);
    else k_e2_final_pair<1024><<<fgrid, 1024, 0, st>>>(a, e, x);
    *launches += 2;
    PD_CUDA(c, cudaGetLastError());
    return 0;
}

// overflow of the interleaved read-pair copies during the last scan? (exact need in *need_words)
int pd_em2_overflow(pd_ctx * c, bool * ovf, size_t * need_words)
{
    *ovf = false; *need_words = 0;
    if (!c->d_scratch[PD_S_E2_CNT]) return 0;
    uint32_t h[2] = {0, 0};
    PD_CUDA(c, cudaMemcpy(h, c->d_scratch[PD_S_E2_CNT], 8, cudaMemcpyDeviceToHost));
    *ovf = h[1] != 0; *need_words = h[0];
    return 0;
}
