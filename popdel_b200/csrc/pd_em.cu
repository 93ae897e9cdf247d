// pd_em.cu -- K3-K5: genotyping of every (flagged window, initial deletion length) pair.
//
//   k_em      one block per pair: initialize_allele_frequency (genotype_deletion_popdel_call.h:93-133), then the EM
//             over deletion length / reference shifts / allele frequency (:556-664). LPS lanes of a warp share one
//             sample (read pairs strided over the lanes, fixed-order shuffle reductions -> deterministic). Loop state
//             (length, frequency, genotype priors, iteration) is kept redundantly in registers by every thread, so an
//             iteration costs two block barriers. Per read pair the insert-size deviation and the posterior weight
//             r = del/(del+ref) of the last data-likelihood pass are cached in shared memory for the length update.
//   k_final   one block per surviving pair: final data likelihoods (:255-337), log10 genotype likelihoods -> PL
//             (utils_popdel.h:1511-1528), LAD/DAD (:137-172), FL, supporting read-pair percentiles (:514-529), LR test.
//   k_em_one  both fused, for cohorts with one read group per sample that fit one block (one sample per lane).
//   k_em_xr / k_final_xr  the general kernels as persistent ticketed blocks with in-kernel cross-rank reductions
//             (sample-sharded cohorts, pd_shard.cu / pd_em_common.cuh).
//   k_emit_stream  concurrent with the EM launch: copies finished pairs (done flags) in pair order into mapped host
//             memory.
// Floating point: double. The two places where the reference's x87 long double is observable are emulated
// (finish_triple): exp() underflow at -11399.5 and the ln2 - fl64(ln2) residue of read pairs with ref == del.
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>

#include "pd_em_common.cuh"

#ifdef PD_EM_STATS
__device__ unsigned long long g_em_stats[32];
#define ST_ADD(i, v) atomicAdd(&g_em_stats[i], (unsigned long long)(v))
#define ST_T0 const long long st_t0_ = clock64()
#define ST_CLK(i, t0) do { if (threadIdx.x == 0) ST_ADD(i, clock64() - (t0)); } while (0)
#else
#define ST_ADD(i, v) do {} while (0)
#define ST_CLK(i, t0) do {} while (0)
#endif

namespace {

// data likelihoods of every sample for (L, shifts) -> dlx (log domain) / dle (exp domain);
// compute_data_likelihoods (EM overload) :179-253. Returns this thread's part of update_allele_frequency's sum
// (:467-485) under the genotype priors `gtf`.
template <int LPS, int SLOTS>
__device__ __forceinline__ double compute_dl(const PdDev & a, const EmArgs & e, EmShared & sh, const uint32_t * cnt, const uint32_t * off,
                                             double * dlx, double * dle, const int32_t * shifts, bool zero_shifts, int L,
                                             double * cache_r, const int32_t * cache_d, bool fill_cache, const Gt gtf, const bool own0)
{
    double fs = 0;
    const int tid = threadIdx.x, T = blockDim.x, sub = tid % LPS, grp = tid / LPS, ngrp = T / LPS;
    const uint32_t gmask = group_mask<LPS>();
    int slot = 0;
    for (uint32_t s = grp; s < a.N; s += ngrp) {
        double l0 = 0, l1 = 0, l2 = 0;
        uint32_t nd = 0;
        for (uint32_t g = a.sample_rg[s]; g < a.sample_rg[s + 1]; ++g) {
            const RgLite k = rg_lite(a.rgc + g);
            const uint32_t n = cnt[g];
            if (n >= k.max_load) {
                if (g == 0 && own0 && sub == 0) sh.rgw[0] = sh.rgw[1] = sh.rgw[2] = 0;      // Triple(0,0,0) in the reference
                continue;
            }
            const int shift = zero_shifts ? 0 : shifts[g];
            const int32_t * p = e.pool_dev + off[g];
            for (uint32_t i = sub; i < n; i += LPS, ++slot) {
                const int d = slot < SLOTS ? cache_d[slot * T + tid] : __ldg(p + i);
                const PdTab * tr = tab_at(a.tab, k, d - shift);
                const D4 rr = ld4(&tr->val);                                 // ref, ln ref, ln(ref + floor) - ln 2, floor / (floor + ref)
                double g1, g2, r;
                if (!tab_in(k, d - L)) {                                     // deletion hypothesis on the floor: the bulk
                    g2 = k.ln_min_prob;
                    if (rr.a == k.min_prob) { g1 = rr.b; ++nd; r = 0.5; }    // ref == del: + LN2_RESIDUE in finish_triple
                    else { g1 = rr.c; r = rr.d; }
                } else {
                    const PdTab * td = a.tab + k.hist_off + (d - L + k.hist_base + 1);
                    const double2 dv = ld2(&td->val);                       // del, ln del
                    g2 = dv.y;
                    if (rr.a == dv.x) { g1 = rr.b; ++nd; r = 0.5; }
                    else if (dv.x == k.min_prob) { g1 = rr.c; r = rr.d; }
                    else if (rr.a == k.min_prob) { const double2 dp = ld2(&td->lnp); g1 = dp.x; r = 1.0 - dp.y; }
                    else { g1 = log(rr.a + dv.x) - LN2_D; r = dv.x / (dv.x + rr.a); }
                }
                if (fill_cache && slot < SLOTS) cache_r[slot * T + tid] = r;
                l0 += rr.b; l1 += g1; l2 += g2;
            }
            if (g == 0 && own0) {                                        // read group 0 = first read group of sample 0 of the cohort
                const double w0 = group_sum<LPS>(l0, gmask), w1 = group_sum<LPS>(l1, gmask), w2 = group_sum<LPS>(l2, gmask);
                if (sub == 0) { const double m = fmax(fmax(w0, w1), w2); sh.rgw[0] = exp(w0 - m); sh.rgw[1] = exp(w1 - m); sh.rgw[2] = exp(w2 - m); }
            }
        }
        l0 = group_sum<LPS>(l0, gmask); l1 = group_sum<LPS>(l1, gmask); l2 = group_sum<LPS>(l2, gmask); nd = group_sum<LPS>(nd, gmask);
        double x0, x1, x2, E0, E1, E2;
        finish_triple(l0, l1, l2, nd, x0, x1, x2);
        if (LPS >= 4) {                                                  // one exp per lane instead of three in a row
            const double xi = sub == 0 ? x0 : (sub == 1 ? x1 : x2);
            const double Ei = xi == 0 ? 1.0 : exp(xi);
            E0 = __shfl_sync(gmask, Ei, 0, LPS); E1 = __shfl_sync(gmask, Ei, 1, LPS); E2 = __shfl_sync(gmask, Ei, 2, LPS);
        } else {
            E0 = x0 == 0 ? 1.0 : exp(x0); E1 = x1 == 0 ? 1.0 : exp(x1); E2 = x2 == 0 ? 1.0 : exp(x2);
        }
        if (sub == 0) {
            dlx[3 * s] = x0; dlx[3 * s + 1] = x1; dlx[3 * s + 2] = x2;
            dle[3 * s] = E0; dle[3 * s + 1] = E1; dle[3 * s + 2] = E2;
            const double p0 = E0 * gtf.a, p1 = E1 * gtf.b, p2 = E2 * gtf.c;
            fs += (p1 + 2 * p2) / (p0 + p1 + p2);
        }
    }
    return fs;
}

// deletion_likelihood_ratio :490-508 (block-wide; result on all threads)
template <bool XR>
__device__ __forceinline__ double block_lr(const PdDev & a, const EmArgs & e, XrBlock & xb, EmShared & sh, const double * dlx, const double * dle, const Gt gt, int & par)
{
    double del = 0, nodel = 0;
    for (uint32_t s = threadIdx.x; s < a.N; s += blockDim.x) {
        const double A = dle[3 * s], B = dle[3 * s + 1], C = dle[3 * s + 2];
        const double p0 = A * gt.a, p1 = B * gt.b, p2 = C * gt.c, pAll = p0 + p1 + p2;
        const double a0 = p0 / pAll, a1 = p1 / pAll, a2 = p2 / pAll;
        del += log(a0 * A + a1 * B + a2 * C);
        nodel += dlx[3 * s];
    }
    block_sum2(del, nodel, sh.red, par);
    if (XR) xr_sum2(e.xr, xb, sh, del, nodel);
    return del - nodel;
}

template <int LPS, int SLOTS, bool XR>
__device__ __forceinline__ void em_body(const PdDev & a, const EmArgs & e, EmShared & sh, double * cache_r, const uint32_t bid)
{
    const int tid = threadIdx.x, T = blockDim.x, sub = tid % LPS, grp = tid / LPS, ngrp = T / LPS;
    int32_t * cache_d = reinterpret_cast<int32_t *>(cache_r + (size_t)SLOTS * T);
    const uint32_t pi = e.pair0 + bid;
    const PdPair pr = e.pairs[pi];
    const uint32_t job = pr.job - e.job_base;
    const int L0 = pr.L0;
    const uint32_t w = e.job_window[pr.job];
    const uint32_t cj = e.cjob_of[job] - e.cj_base;
    const uint32_t * cnt = e.act_cnt + (size_t)cj * a.R;
    const uint32_t * off = e.act_off + (size_t)cj * a.R;
    double * dlx = e.dlx + (size_t)bid * 3 * a.N;
    double * dle = e.dle + (size_t)bid * 3 * a.N;
    int32_t * shifts = e.shifts + (size_t)bid * a.R;
    const uint32_t gmask = group_mask<LPS>();
    int par = 0;
    XrBlock xb{bid, e.xr.epoch << 16};
    const bool own0 = !XR || e.xr.owns_rg0;             // read group 0 of the cohort lives on this rank
    const double n_cohort = XR ? (double)e.xr.n_global : (double)a.N;
    // loop state, identical on every thread
    uint32_t len = (uint32_t)L0, it = 0;
    double freq = 0;
    Gt gt = Gt{1, 0, 0};
    auto finish = [&](uint32_t alive, uint32_t reason) {
        if (tid == 0) {
            EmState st; st.len = len; st.it = it; st.alive = alive; st.pad = 0; st.freq = freq;
            st.gt[0] = gt.a; st.gt[1] = gt.b; st.gt[2] = gt.c;
            e.states[bid] = st;
            if (!alive) {
                e.valid[bid] = 0;
                if (e.dbg) { e.dbg[4 * bid] = reason; e.dbg[4 * bid + 1] = len; e.dbg[4 * bid + 2] = it; }
            }
        }
    };

    for (uint32_t g = tid; g < a.R; g += T) shifts[g] = 0;
    if (tid == 0) sh.nvisited = 0;

    // ---- initialize_allele_frequency :93-133 (also fills the deviation cache)
    {
        unsigned long long c = 0, t = 0;
        int slot = 0;
        for (uint32_t s = grp; s < a.N; s += ngrp)
            for (uint32_t g = a.sample_rg[s]; g < a.sample_rg[s + 1]; ++g) {
                const uint32_t n = cnt[g];
                if (n >= __ldg(&a.rgc[g].max_load)) continue;
                if (sub == 0) t += n;
                const double sd = __ldg(&a.rgc[g].stddev);
                const int wb = max(L0 / 2, (int)floor((double)L0 - 2 * sd + 0.5));
                const int we = (int)((double)L0 + 2 * sd);
                const int32_t * p = e.pool_dev + off[g];
                for (uint32_t i = sub; i < n; i += LPS, ++slot) {
                    const int d = __ldg(p + i);
                    if (slot < SLOTS) cache_d[slot * T + tid] = d;
                    c += (d > wb && d < we);
                }
            }
        block_sum2u(c, t, sh.redu);
        if (XR) xr_sum2u(e.xr, xb, sh, c, t);
        freq = t == 0 ? 0.0 : (double)c / (double)t;
        gt = gt_prior(freq, e.somatic);
    }
    if (freq == 0) { finish(0, 1); return; }
    compute_dl<LPS, SLOTS>(a, e, sh, cnt, off, dlx, dle, shifts, true, L0, cache_r, cache_d, true, gt, own0);
    __syncthreads();
    if (XR) {                                           // read group 0's likelihood triple comes from its owner
        double z = 0, r0 = own0 ? sh.rgw[0] : 0.0, r1 = own0 ? sh.rgw[1] : 0.0, r2 = own0 ? sh.rgw[2] : 0.0;
        xr_sum4(e.xr, xb, sh, z, r0, r1, r2);
        if (tid == 0) { sh.rgw[0] = r0; sh.rgw[1] = r1; sh.rgw[2] = r2; }
        __syncthreads();
    }

    // ---- EM loop :598-660
    uint32_t prevLen = len; double prevFreq = freq;
    int stop = 0;
    while (len >= e.min_len && it < e.iterations) {
        ++it;
        prevLen = len; prevFreq = freq;
        // posterior weights of read group 0 (rgDlIt is never advanced, :401,424-431)
        const double r0 = sh.rgw[0], r1 = sh.rgw[1], r2 = sh.rgw[2];
        const double aSumRg = r0 * gt.a + r1 * gt.b + r2 * gt.c;
        const double ea0Rg = r0 * gt.a / aSumRg, ea1Rg = r1 * gt.b / aSumRg;      // NaN when read group 0 is high-coverage
        // update_deletion_length :388-462
        const int L = (int)len;
        double sumDel = 0, wDel = 0;
        {
            int slot = 0;
            for (uint32_t s = grp; s < a.N; s += ngrp) {
                const double E1 = dle[3 * s + 1], E2 = dle[3 * s + 2];
                const double inv = 1.0 / (dle[3 * s] * gt.a + E1 * gt.b + E2 * gt.c);
                const double ea1 = E1 * gt.b * inv, ea2 = E2 * gt.c * inv;
                for (uint32_t g = a.sample_rg[s]; g < a.sample_rg[s + 1]; ++g) {
                    const uint32_t n = cnt[g];
                    if (n >= __ldg(&a.rgc[g].max_load)) continue;
                    double sumRef = 0, wRef = 0;
                    const int32_t * p = e.pool_dev + off[g];
                    for (uint32_t i = sub; i < n; i += LPS, ++slot) {
                        int d; double r;
                        if (slot < SLOTS) { d = cache_d[slot * T + tid]; r = cache_r[slot * T + tid]; }
                        else { d = __ldg(p + i); r = pair_weight(a.tab, rg_lite(a.rgc + g), d, shifts[g], L); }
                        const double pd = ea1 * r + ea2;
                        const double prf = ea1Rg * (1.0 - r) + ea0Rg;
                        sumDel += pd; sumRef += prf;
                        wDel += pd * d; wRef += prf * d;
                    }
                    sumRef = group_sum<LPS>(sumRef, gmask); wRef = group_sum<LPS>(wRef, gmask);
                    if (sub == 0) {
                        const double q = wRef / sumRef;
                        int sft = (q != q) ? 0 : (q >= 2147483647.0 ? INT_MAX : (q <= -2147483648.0 ? INT_MIN : (int)q));
                        const double sd = __ldg(&a.rgc[g].stddev);
                        if (sft > sd || sft < -1 * sd) sft = 0;
                        shifts[g] = sft;
                    }
                }
            }
        }
        block_sum2(sumDel, wDel, sh.red, par);
        if (XR) xr_sum2(e.xr, xb, sh, sumDel, wDel);
        if (tid == 0) {                                   // visited[prevLen] = prevFreq (:600); read after the next barrier
            int f = -1;
            for (int i = 0; i < sh.nvisited; ++i) if (sh.visited_len[i] == (int)prevLen) f = i;
            if (f < 0) { f = sh.nvisited++; sh.visited_len[f] = (int)prevLen; }
            sh.visited_freq[f] = prevFreq;
            if ((int)w == e.dbg_window)
                printf("GPU w %u L0 %d it %u len %u freq %.17g sumDel %.17g wDel %.17g\n", w, L0, it, len, freq, sumDel, wDel);
        }
        if (sumDel == 0) len = 0;
        else { const double nl = wDel / sumDel; len = nl < 0 ? 0u : (uint32_t)round(nl); }
        // data likelihoods at the new length + update_allele_frequency :467-485 (priors of the previous iteration)
        double fs = compute_dl<LPS, SLOTS>(a, e, sh, cnt, off, dlx, dle, shifts, false, (int)len, cache_r, cache_d, true, gt, own0), dummy = 0;
        block_sum2(fs, dummy, sh.red, par);
        if (XR) {
            double r0 = own0 ? sh.rgw[0] : 0.0, r1 = own0 ? sh.rgw[1] : 0.0, r2 = own0 ? sh.rgw[2] : 0.0;
            xr_sum4(e.xr, xb, sh, fs, r0, r1, r2);
            if (tid == 0) { sh.rgw[0] = r0; sh.rgw[1] = r1; sh.rgw[2] = r2; }
            __syncthreads();
        }
        freq = fs / 2.0 / n_cohort;
        if (freq == 0) { stop = 1; break; }
        gt = gt_prior(freq, e.somatic);
        for (int i = 0; i < sh.nvisited; ++i)
            if (sh.visited_len[i] == (int)len && fabs(sh.visited_freq[i] - freq) <= 0.0001) stop = 2;
        if (stop == 2) {
            // convergence :632-658: compare with the previous estimate evaluated with the initial (zero) shifts
            const double lr = block_lr<XR>(a, e, xb, sh, dlx, dle, gt, par);
            const Gt prevGt = gt_prior(prevFreq, e.somatic);          // the priors the previous estimate was made with
            compute_dl<LPS, SLOTS>(a, e, sh, cnt, off, dlx, dle, shifts, true, (int)prevLen, cache_r, cache_d, false, prevGt, own0);
            __syncthreads();
            const double plr = block_lr<XR>(a, e, xb, sh, dlx, dle, prevGt, par);
            if (plr > lr) {
                len = prevLen; freq = prevFreq;
                for (uint32_t g = tid; g < a.R; g += T) shifts[g] = 0;
            }
            break;
        }
    }
    const bool alive = !(freq < 0.0000000001 || len < e.min_len);
    finish(alive ? 1u : 0u, 2);
}

template <int LPS, int SLOTS, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB) k_em(PdDev a, EmArgs e)
{
    __shared__ EmShared sh;
    extern __shared__ double cache_r[];                 // [SLOTS][T] weights, then [SLOTS][T] deviations (int32)
    em_body<LPS, SLOTS, false>(a, e, sh, cache_r, blockIdx.x);
}
// sample-sharded cohort: persistent blocks take the pairs in ticket order, so that the pairs in flight are the same
// (lowest unfinished) ones on every rank and the in-kernel exchanges cannot wait for a block that is not resident
template <int LPS, int SLOTS, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB) k_em_xr(PdDev a, EmArgs e)
{
    __shared__ EmShared sh;
    __shared__ uint32_t s_bid;
    extern __shared__ double cache_r[];
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_bid = atomicAdd(e.xr.ticket, 1u);
        __syncthreads();
        const uint32_t bid = s_bid;
        if (bid >= e.npairs) return;
        em_body<LPS, SLOTS, true>(a, e, sh, cache_r, bid);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// final pass: one block per (window, initial length) that survived the EM
// ------------------------------------------------------------------------------------------------------------------
constexpr uint32_t SUPP_CAP = 1536;                    // supporting read pairs kept in shared memory for the percentiles

template <int LPS, bool XR>
__device__ __forceinline__ void final_body(const PdDev & a, const EmArgs & e, EmShared & sh, uint32_t * s_first, uint32_t * s_last, uint32_t & s_nsupp,
                                           const uint32_t bid)
{
    const EmState stt = e.states[bid];
    XrBlock xb{bid, e.xr.epoch << 16};
    if (XR && bid == 0) {
        // one exchange per launch even when no pair survived the EM: a rank that has passed this launch then knows that
        // every peer has left the previous one, whose slots the next launch reuses
        unsigned long long z0 = 0, z1 = 0;
        xr_sum2u(e.xr, xb, sh, z0, z1);
    }
    if (!stt.alive) return;
    const double n_cohort = XR ? (double)e.xr.n_global : (double)a.N;
    const int tid = threadIdx.x, T = blockDim.x, sub = tid % LPS, grp = tid / LPS, ngrp = T / LPS;
    const uint32_t gmask = group_mask<LPS>();
    if (tid == 0) s_nsupp = 0;
    const uint32_t pi = e.pair0 + bid;
    const PdPair pr = e.pairs[pi];
    const uint32_t job = pr.job - e.job_base;
    const uint32_t L0 = (uint32_t)pr.L0;
    const uint32_t w = e.job_window[pr.job];
    const uint32_t cj = e.cjob_of[job] - e.cj_base;
    const uint32_t * cnt = e.act_cnt + (size_t)cj * a.R;
    const uint32_t * off = e.act_off + (size_t)cj * a.R;
    const uint8_t * sstat = e.sstat + (size_t)job * a.N;
    double * dlx = e.dlx + (size_t)bid * 3 * a.N;
    double * dle = e.dle + (size_t)bid * 3 * a.N;
    const int32_t * shifts = e.shifts + (size_t)bid * a.R;
    uint32_t * ps = e.ps + (size_t)bid * 13 * a.N;
    const int len = (int)stt.len;
    const Gt gt = Gt{stt.gt[0], stt.gt[1], stt.gt[2]};
    int par = 0;
    __syncthreads();
    auto reject = [&](uint32_t reason) {
        if (tid == 0) {
            e.valid[bid] = 0;
            if (e.dbg) { e.dbg[4 * bid] = reason; e.dbg[4 * bid + 1] = stt.len; e.dbg[4 * bid + 2] = stt.it; }
        }
    };
    // ---- final pass :665-727 (compute_data_likelihoods final overload :255-337)
    unsigned long long supp = 0, ndata = 0;
    uint32_t smin = 0xFFFFFFFFu, smax = 0, lmin = 0xFFFFFFFFu, lmax = 0;   // ranges of supporting starts / ends
    for (uint32_t s = grp; s < a.N; s += ngrp) {
        uint32_t lad0 = 0, lad1 = 0, lad2 = 0, dad0 = 0, dad1 = 0, dad2 = 0, dad3 = 0, dad4 = 0;
        uint32_t fl_min = 0xFFFFFFFFu, fl_max = 0, ndeg = 0;
        double l0 = 0, l1 = 0, l2 = 0, t0 = 0, t1 = 0, t2 = 0;
        int delLower = INT_MAX, delUpper = 0;
        const uint32_t g0 = a.sample_rg[s], g1 = a.sample_rg[s + 1];
        for (uint32_t g = g0; g < g1; ++g) {
            const PdRgConst k = a.rgc[g];
            const uint32_t n = cnt[g];
            if (n >= k.max_load) continue;
            const int shift = shifts[g];
            delLower = len - k.lower_q; delUpper = len + k.upper_q;
            const uint32_t * pp = e.pool_pos + off[g];
            const int32_t * pd = e.pool_dev + off[g];
            for (uint32_t i = sub; i < n; i += LPS) {
                const int d = __ldg(pd + i);
                if (d > k.upper_q) { if (d < delLower) ++dad2; else if (d <= delUpper) ++dad3; else ++dad4; }
                else { if (d < delUpper) ++dad0; else ++dad1; }
                const PdTab * tr = tab_at(a.tab, k, d - shift);
                const PdTab * td = tab_at(a.tab, k, d - len);
                const D4 r1 = ld4(&tr->val), r2 = ld4(&tr->l10);                              // full row: two 256-bit loads
                D4 d1 = D4{k.min_prob, k.ln_min_prob, 0, 0}, d2 = D4{k.l10_min_prob, 0, 0, 0};    // floor: .c / .b unused
                if (td != a.tab + k.hist_off) { d1 = ld4(&td->val); d2 = ld4(&td->l10); }
                const double ref = r1.a, del = d1.a;
                if (ref >= 2 * del) ++lad0; else if (del >= 2 * ref) ++lad2; else ++lad1;
                l0 += r1.b; t0 += r2.a;
                l2 += d1.b; t2 += d2.a;
                if (ref == del) { l1 += r1.b; t1 += r2.a; ++ndeg; }                          // residues applied below
                else if (del == k.min_prob) { l1 += r1.c; t1 += r2.b; }
                else if (ref == k.min_prob) { l1 += d1.c; t1 += d2.b; }
                else { l1 += log(ref + del) - LN2_D; t1 += log10(ref + del) - LOG10_2_D; }
                const uint32_t first = __ldg(pp + i) + e.anchor;
                const uint32_t last = first + (uint32_t)max(0, d + k.inner_off);
                fl_min = min(fl_min, first); fl_max = max(fl_max, last);
            }
        }
        // supporting read pairs: borders of the LAST usable read group apply to all of the sample's read groups (quirk)
        for (uint32_t g = g0; g < g1; ++g) {
            const uint32_t n = cnt[g];
            if (n >= __ldg(&a.rgc[g].max_load)) continue;
            const int inner_off = __ldg(&a.rgc[g].inner_off);
            const uint32_t * pp = e.pool_pos + off[g];
            const int32_t * pd = e.pool_dev + off[g];
            for (uint32_t i = sub; i < n; i += LPS) {
                const int d = __ldg(pd + i);
                if (d >= delLower && d <= delUpper) {
                    const uint32_t first = __ldg(pp + i) + e.anchor;
                    const uint32_t last = first + (uint32_t)max(0, d + inner_off);
                    ++supp; smin = min(smin, first); smax = max(smax, first); lmin = min(lmin, last); lmax = max(lmax, last);
                    const uint32_t slot = atomicAdd(&s_nsupp, 1u);
                    if (slot < SUPP_CAP) { s_first[slot] = first; s_last[slot] = last; }
                }
            }
        }
        lad0 = group_sum<LPS>(lad0, gmask); lad1 = group_sum<LPS>(lad1, gmask); lad2 = group_sum<LPS>(lad2, gmask);
        dad0 = group_sum<LPS>(dad0, gmask); dad1 = group_sum<LPS>(dad1, gmask); dad2 = group_sum<LPS>(dad2, gmask);
        dad3 = group_sum<LPS>(dad3, gmask); dad4 = group_sum<LPS>(dad4, gmask); ndeg = group_sum<LPS>(ndeg, gmask);
        fl_min = group_min<LPS>(fl_min, gmask); fl_max = group_max<LPS>(fl_max, gmask);
        l0 = group_sum<LPS>(l0, gmask); l1 = group_sum<LPS>(l1, gmask); l2 = group_sum<LPS>(l2, gmask);
        t0 = group_sum<LPS>(t0, gmask); t1 = group_sum<LPS>(t1, gmask); t2 = group_sum<LPS>(t2, gmask);
        if (sub != 0) continue;
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
        dlx[3 * s] = x0; dlx[3 * s + 1] = x1; dlx[3 * s + 2] = x2;
        dle[3 * s] = exp(x0); dle[3 * s + 1] = exp(x1); dle[3 * s + 2] = exp(x2);
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
    }
    __syncthreads();
    block_sum2u(supp, ndata, sh.redu);
    if (XR) xr_sum2u(e.xr, xb, sh, supp, ndata);
    if (supp == 0) { reject(3); return; }
    // percentiles of the supporting starts (80th) and ends (20th): getSuppFirstLast :514-529, by value bisection
    uint32_t sF, sL;
    const unsigned long long kF = (unsigned long long)round((double)(supp - 1) * 0.8);
    const unsigned long long kL = (unsigned long long)round((double)(supp - 1) * (1 - 0.8));
    if (!XR && supp <= SUPP_CAP) {
        // the usual case: the supporting read pairs sit in shared memory and one warp bisects without block barriers
        if (tid < 32) {
            const uint32_t n = (uint32_t)supp;
            uint32_t loF = 0xFFFFFFFFu, hiF = 0, loL = 0xFFFFFFFFu, hiL = 0;
            for (uint32_t i = tid; i < n; i += 32) { loF = min(loF, s_first[i]); hiF = max(hiF, s_first[i]); loL = min(loL, s_last[i]); hiL = max(hiL, s_last[i]); }
            for (int o = 16; o > 0; o >>= 1) {
                loF = min(loF, __shfl_xor_sync(PD_FULL, loF, o)); hiF = max(hiF, __shfl_xor_sync(PD_FULL, hiF, o));
                loL = min(loL, __shfl_xor_sync(PD_FULL, loL, o)); hiL = max(hiL, __shfl_xor_sync(PD_FULL, hiL, o));
            }
            while (loF < hiF || loL < hiL) {
                const uint32_t midF = loF + (hiF - loF) / 2, midL = loL + (hiL - loL) / 2;
                uint32_t cF = 0, cL = 0;
                for (uint32_t i = tid; i < n; i += 32) { cF += s_first[i] <= midF; cL += s_last[i] <= midL; }
                for (int o = 16; o > 0; o >>= 1) { cF += __shfl_xor_sync(PD_FULL, cF, o); cL += __shfl_xor_sync(PD_FULL, cL, o); }
                if (loF < hiF) { if (cF >= kF + 1) hiF = midF; else loF = midF + 1; }
                if (loL < hiL) { if (cL >= kL + 1) hiL = midL; else loL = midL + 1; }
            }
            if (tid == 0) { sh.sel[0] = loF; sh.sel[1] = loL; }
        }
        __syncthreads();
        sF = sh.sel[0]; sL = sh.sel[1];
    } else {
        // block-wide min/max of the supporting positions (shuffles, then warps in index order)
        for (int o = 16; o > 0; o >>= 1) {
            smin = min(smin, __shfl_xor_sync(PD_FULL, smin, o)); smax = max(smax, __shfl_xor_sync(PD_FULL, smax, o));
            lmin = min(lmin, __shfl_xor_sync(PD_FULL, lmin, o)); lmax = max(lmax, __shfl_xor_sync(PD_FULL, lmax, o));
        }
        uint32_t * r32 = reinterpret_cast<uint32_t *>(sh.red);
        const int wid = tid >> 5, nw = (T + 31) >> 5;
        __syncthreads();
        if ((tid & 31) == 0) { r32[4 * wid] = smin; r32[4 * wid + 1] = smax; r32[4 * wid + 2] = lmin; r32[4 * wid + 3] = lmax; }
        __syncthreads();
        for (int i = 0; i < nw; ++i) { smin = min(smin, r32[4 * i]); smax = max(smax, r32[4 * i + 1]); lmin = min(lmin, r32[4 * i + 2]); lmax = max(lmax, r32[4 * i + 3]); }
        __syncthreads();
        if (XR) xr_minmax(e.xr, xb, sh, smin, smax, lmin, lmax);
        uint32_t loF = smin, hiF = smax, loL = lmin, hiL = lmax;
        while (loF < hiF || loL < hiL) {
            const uint32_t midF = loF + (hiF - loF) / 2, midL = loL + (hiL - loL) / 2;
            unsigned long long cF = 0, cL = 0;
            for (uint32_t s = tid; s < a.N; s += T) {
                int delLower = INT_MAX, delUpper = 0;
                const uint32_t g0 = a.sample_rg[s], g1 = a.sample_rg[s + 1];
                for (uint32_t g = g0; g < g1; ++g) { const PdRgConst k = a.rgc[g]; if (cnt[g] >= k.max_load) continue; delLower = len - k.lower_q; delUpper = len + k.upper_q; }
                for (uint32_t g = g0; g < g1; ++g) {
                    const PdRgConst k = a.rgc[g];
                    const uint32_t n = cnt[g];
                    if (n >= k.max_load) continue;
                    const uint32_t * pp = e.pool_pos + off[g];
                    const int32_t * pd = e.pool_dev + off[g];
                    for (uint32_t i = 0; i < n; ++i) {
                        const int d = pd[i];
                        if (d >= delLower && d <= delUpper) {
                            const uint32_t first = pp[i] + e.anchor;
                            const uint32_t last = first + (uint32_t)max(0, d + k.inner_off);
                            cF += first <= midF; cL += last <= midL;
                        }
                    }
                }
            }
            block_sum2u(cF, cL, sh.redu);
            if (XR) xr_sum2u(e.xr, xb, sh, cF, cL);
            if (loF < hiF) { if (cF >= kF + 1) hiF = midF; else loF = midF + 1; }
            if (loL < hiL) { if (cL >= kL + 1) hiL = midL; else loL = midL + 1; }
        }
        sF = loF; sL = loL;
    }
    if (sF == 0 && sL == 0) { reject(4); return; }
    const double lr = block_lr<XR>(a, e, xb, sh, dlx, dle, gt, par);
    if (tid == 0) {
        const bool ok = lr >= e.min_lr;
        e.valid[bid] = ok ? 1 : 0;
        if (e.dbg) { e.dbg[4 * bid] = ok ? 0 : 5; e.dbg[4 * bid + 1] = stt.len; e.dbg[4 * bid + 2] = stt.it; e.dbg[4 * bid + 3] = (uint32_t)supp; }
        if (ok) {
            pd_call c;
            c.initial_length = L0; c.iterations = stt.it; c.deletion_length = stt.len;
            c.filter = ((double)ndata / n_cohort >= e.min_sample_fraction) ? 0u : 4u;
            c.lr = lr; c.frequency = stt.freq;
            const uint32_t cur = e.anchor + w * PD_WIN;
            c.window_position = cur - 1;
            c.position = e.window_wise ? cur - 1 : sF;
            c.end_position = e.window_wise ? 0u : sL;
            c.segment = (uint32_t)(((uint64_t)w * PD_WIN) / a.window_buffer);
            e.calls[bid] = c;
        }
    }
}

template <int LPS, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB) k_final(PdDev a, EmArgs e)
{
    __shared__ EmShared sh;
    __shared__ uint32_t s_first[SUPP_CAP], s_last[SUPP_CAP];
    __shared__ uint32_t s_nsupp;
    final_body<LPS, false>(a, e, sh, s_first, s_last, s_nsupp, blockIdx.x);
    publish_done(e, blockIdx.x);
}
template <int LPS, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB) k_final_xr(PdDev a, EmArgs e)
{
    __shared__ EmShared sh;
    __shared__ uint32_t s_first[SUPP_CAP], s_last[SUPP_CAP];
    __shared__ uint32_t s_nsupp, s_bid;
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_bid = atomicAdd(e.xr.ticket + 1, 1u);
        __syncthreads();
        const uint32_t bid = s_bid;
        if (bid >= e.npairs) return;
        final_body<LPS, true>(a, e, sh, s_first, s_last, s_nsupp, bid);
        publish_done(e, bid);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Fused EM + final pass for cohorts with ONE read group per sample that fit one block (N <= blockDim / LPS): every
// lane group owns one sample for the whole kernel, so the per-sample state (table constants, reference shift, data
// likelihoods, posterior-weight moments) lives in registers and only the table look-ups touch memory. The look-ups of
// four read pairs are issued together to overlap their L2 latency. The length update needs no pass over the read
// pairs: with r_i = del_i / (del_i + ref_i) from the last data-likelihood pass,
//     sum_i p_del,i = ea1 * sum r_i + n * ea2           sum_i p_del,i * d_i = ea1 * sum r_i d_i + ea2 * sum d_i
// (update_deletion_length :388-462), likewise for the reference weights.
// ------------------------------------------------------------------------------------------------------------------
struct RgOne { const PdTab * fl; int hist_base; uint32_t hist_len; double min_prob, ln_min_prob; };   // fl = floor row of the read group

template <int LPS, int SLOTS, int BATCH>
__device__ __forceinline__ void dl_one(const RgOne & k, const int32_t * cache_d, const int32_t * pd,
                                       int T, int tid, int sub, int nl, int shift, int L, uint32_t gmask, double * rgw /* group of read group 0 only */,
                                       double & x0, double & E0, double & E1, double & E2, double & Sr, double & Srd)
{
    double l0 = 0, l1 = 0, l2 = 0, sr = 0, srd = 0;
    uint32_t nd = 0;
    const PdTab * fl = k.fl;
    for (int b = 0; b < nl; b += BATCH) {
        int d[BATCH]; uint32_t id[BATCH]; D4 rr[BATCH]; double2 dv[BATCH];
#pragma unroll
        for (int j = 0; j < BATCH; ++j) {                            // BATCH independent pairs of look-ups in flight
            const int jj = b + j;
            const bool v = jj < nl;
            d[j] = v ? (jj < SLOTS ? cache_d[jj * T + tid] : __ldg(pd + sub + jj * LPS)) : 0;
            const uint32_t ir = v && tab_in(k, d[j] - shift) ? (uint32_t)(d[j] - shift + k.hist_base + 1) : 0u;
            id[j] = v && tab_in(k, d[j] - L) ? (uint32_t)(d[j] - L + k.hist_base + 1) : 0u;
            rr[j] = ld4(&fl[ir].val);                                // ref, ln ref, ln(ref + floor) - ln 2, floor / (floor + ref)
            dv[j] = make_double2(k.min_prob, k.ln_min_prob);         // deletion hypothesis below the histogram: the bulk
            if (id[j]) dv[j] = ld2(&fl[id[j]].val);
        }
#pragma unroll
        for (int j = 0; j < BATCH; ++j) {
            if (b + j >= nl) break;
            const double ref = rr[j].a, del = dv[j].x;
            double g1, r;
            if (ref == del) { g1 = rr[j].b; ++nd; r = 0.5; }                 // + LN2_RESIDUE in finish_triple
            else if (del == k.min_prob) { g1 = rr[j].c; r = rr[j].d; }
            else if (ref == k.min_prob) { const double2 dp = ld2(&fl[id[j]].lnp); g1 = dp.x; r = 1.0 - dp.y; }
            else { g1 = log(ref + del) - LN2_D; r = del / (del + ref); }
            l0 += rr[j].b; l1 += g1; l2 += dv[j].y;
            sr += r; srd += r * d[j];
        }
    }
    l0 = group_sum<LPS>(l0, gmask); l1 = group_sum<LPS>(l1, gmask); l2 = group_sum<LPS>(l2, gmask);
    Sr = group_sum<LPS>(sr, gmask); Srd = group_sum<LPS>(srd, gmask); nd = group_sum<LPS>(nd, gmask);
    if (rgw && sub == 0) { const double m = fmax(fmax(l0, l1), l2); rgw[0] = exp(l0 - m); rgw[1] = exp(l1 - m); rgw[2] = exp(l2 - m); }
    double x1, x2;
    finish_triple(l0, l1, l2, nd, x0, x1, x2);
    if (LPS >= 4) {                                                  // one exp per lane instead of three in a row
        const double xi = sub == 0 ? x0 : (sub == 1 ? x1 : x2);
        const double Ei = xi == 0 ? 1.0 : exp(xi);
        E0 = __shfl_sync(gmask, Ei, 0, LPS); E1 = __shfl_sync(gmask, Ei, 1, LPS); E2 = __shfl_sync(gmask, Ei, 2, LPS);
    } else {
        E0 = x0 == 0 ? 1.0 : exp(x0); E1 = x1 == 0 ? 1.0 : exp(x1); E2 = x2 == 0 ? 1.0 : exp(x2);
    }
}

// read pairs per lane whose loads the final pass issues together
constexpr int FINAL_BATCH = 2;

template <int LPS, int SLOTS, int BATCH>
__device__ __forceinline__ void em_one_body(const PdDev & a, const EmArgs & e, EmShared & sh, uint32_t * s_first, uint32_t * s_last,
                                            uint32_t & s_nsupp, uint16_t * s_perm, int32_t * cache_dev, double * s_slot)
{
    const int tid = threadIdx.x, T = blockDim.x, sub = tid % LPS;
    const uint32_t gmask = group_mask<LPS>();
    const uint32_t pi = e.pair0 + blockIdx.x;
    const PdPair pr = e.pairs[pi];
    const uint32_t job = pr.job - e.job_base;
    const int L0 = pr.L0;
    const uint32_t w = e.job_window[pr.job];
    int par = 0;
#ifdef PD_EM_STATS
    const long long st_begin = clock64();
    long long st_t = st_begin;
    if (tid == 0) ST_ADD(0, 1);
#endif
    if (tid == 0) { sh.nvisited = 0; s_nsupp = 0; }
    // sample order: by largest deviation, descending, so that the carriers of the deletion share the leading warps and
    // the warps of non-carriers can skip the data-likelihood pass once their reference shift has settled (see below)
    const int32_t * dmx_all = e.dmax + (size_t)job * a.N;
    if (e.sort_samples) {
        for (uint32_t q = tid; q < a.N; q += T) {
            const int32_t v = __ldg(dmx_all + q);
            uint32_t rank = 0;
            for (uint32_t j = 0; j < a.N; ++j) { const int32_t u = __ldg(dmx_all + j); rank += (u > v) || (u == v && j < q); }
            s_perm[rank] = (uint16_t)q;
        }
    }
    __syncthreads();
#ifdef PD_EM_STATS
    ST_CLK(2, st_t); st_t = clock64();
#endif
    const bool has = (uint32_t)(tid / LPS) < a.N;
    const uint32_t s = has ? (e.sort_samples ? s_perm[tid / LPS] : (uint32_t)(tid / LPS)) : 0u;    // my sample = my read group
    const int dmx = has ? __ldg(dmx_all + s) : INT_MIN;

    // ---- per-sample constants and this lane's read pairs
    const PdRgConst * rg = a.rgc + (has ? s : 0);
    RgOne k;
    k.fl = a.tab + __ldg(&rg->hist_off); k.hist_base = __ldg(&rg->hist_base); k.hist_len = __ldg(&rg->hist_len); k.min_prob = __ldg(&rg->min_prob); k.ln_min_prob = __ldg(&rg->ln_min_prob);
    const uint32_t cj = e.cjob_of[job] - e.cj_base;
    const uint32_t n_all = has ? e.act_cnt[(size_t)cj * a.R + s] : 0u;
    const bool usable = has && n_all < __ldg(&rg->max_load);
    const uint32_t n = usable ? n_all : 0u;
    const uint32_t poff = has ? e.act_off[(size_t)cj * a.R + s] : 0u;
    const int32_t * pd = e.pool_dev + poff;
    const int nl = n > (uint32_t)sub ? (int)((n - sub + LPS - 1) / LPS) : 0;
    const double dn = (double)n;

    uint32_t len = (uint32_t)L0, it = 0;
    double freq, Sd;
    Gt gt;
    // ---- initialize_allele_frequency :93-133
    {
        const double sd = __ldg(&a.rgc[has ? s : 0].stddev);
        const int wb = max(L0 / 2, (int)floor((double)L0 - 2 * sd + 0.5));
        const int we = (int)((double)L0 + 2 * sd);
        unsigned long long c = 0, t = sub == 0 ? n : 0u;
        double sdl = 0;
        for (int j = 0; j < nl; ++j) {
            const int d = __ldg(pd + sub + j * LPS);
            if (j < SLOTS) cache_dev[j * T + tid] = d;
            c += (d > wb && d < we);
            sdl += d;
        }
        Sd = group_sum<LPS>(sdl, gmask);
        block_sum2u(c, t, sh.redu);
        freq = t == 0 ? 0.0 : (double)c / (double)t;
        gt = gt_prior(freq, e.somatic);
    }
#ifdef PD_EM_STATS
    ST_CLK(3, st_t); st_t = clock64();
#endif
    if (freq == 0) {
        if (tid == 0) {
            e.valid[blockIdx.x] = 0; if (e.dbg) { e.dbg[4 * blockIdx.x] = 1; e.dbg[4 * blockIdx.x + 1] = len; e.dbg[4 * blockIdx.x + 2] = 0; }
        }
        return;
    }
    int shift = 0;
    double x0, E0, E1, E2, Sr, Srd;
    double * rgw = (has && s == 0 && usable) ? sh.rgw : nullptr;     // read group 0 (quirk: its posterior drives every reference shift)
    if (has && s == 0 && sub == 0 && !usable) sh.rgw[0] = sh.rgw[1] = sh.rgw[2] = 0;      // Triple(0,0,0) in the reference
    auto lr_now = [&](const Gt g) {                      // deletion_likelihood_ratio :490-508
        double del = 0, nodel = 0;
        if (has && sub == 0) {
            const double p0 = E0 * g.a, p1 = E1 * g.b, p2 = E2 * g.c, pAll = p0 + p1 + p2;
            del = log(p0 / pAll * E0 + p1 / pAll * E1 + p2 / pAll * E2);
            nodel = x0;
        }
        block_sum2(del, nodel, sh.red, par);
        return del - nodel;
    };

    // ---- EM loop :598-660 as a small state machine around ONE data-likelihood call site:
    // mode 0 = likelihoods of the initial length, 1 = of an updated length, 2 = of the previous estimate with zero shifts
    uint32_t prevLen = len; double prevFreq = freq, lr_conv = 0;
    int mode = 0, dlL = L0, dlS = 0, curL = INT_MIN, curS = 0;
    for (;;) {
        // A sample whose read pairs all lie below the histogram of the deletion hypothesis at both lengths (dmx) and
        // whose reference shift did not change has exactly the likelihoods and moments it already holds: skip the pass.
        // ... and so does any sample asked for exactly the (length, shift) it was last evaluated with.
        const bool same = e.sort_samples && curL != INT_MIN && dlS == curS &&
                          (dlL == curL || (dmx < dlL - k.hist_base + 1 && dmx < curL - k.hist_base + 1));
#ifdef PD_EM_STATS
        const long long st_p = clock64();
        {
            const uint32_t bm = __ballot_sync(PD_FULL, !same && nl > 0);
            int mx = (!same) ? nl : 0, sm = mx;
            for (int o = 16; o > 0; o >>= 1) { mx = max(mx, __shfl_xor_sync(PD_FULL, mx, o)); sm += __shfl_xor_sync(PD_FULL, sm, o); }
            if ((tid & 31) == 0) { ST_ADD(10, bm != 0); ST_ADD(11, mx); ST_ADD(12, sm); ST_ADD(14 + mode, bm != 0); ST_ADD(17 + mode, sm); }
        }
#endif
        if (mode == 2) {
            // Previous estimate with zero shifts (:641-647). A sample without read pairs inside the deletion histogram at the
            // initial AND the previous length has exactly the likelihoods of the first pass, which are kept in s_slot: swap
            // them in. Every other sample parks its current likelihoods there and recomputes. Either way s_slot then holds
            // what the registers must get back if the newest estimate wins, so the final pass never recomputes the ln sums.
            const bool keep = nl == 0 || (dmx < L0 - k.hist_base + 1 && dmx < dlL - k.hist_base + 1);
            const double a0 = s_slot[tid], a1 = s_slot[T + tid], a2 = s_slot[2 * T + tid], a3 = s_slot[3 * T + tid];
            s_slot[tid] = x0; s_slot[T + tid] = E0; s_slot[2 * T + tid] = E1; s_slot[3 * T + tid] = E2;
            if (keep) { x0 = a0; E0 = a1; E1 = a2; E2 = a3; }
            else dl_one<LPS, SLOTS, BATCH>(k, cache_dev, pd, T, tid, sub, nl, dlS, dlL, gmask, rgw, x0, E0, E1, E2, Sr, Srd);
        } else if (!same) {
            dl_one<LPS, SLOTS, BATCH>(k, cache_dev, pd, T, tid, sub, nl, dlS, dlL, gmask, rgw, x0, E0, E1, E2, Sr, Srd);
            curL = dlL; curS = dlS;
        }
#ifdef PD_EM_STATS
        if (tid == 0) { ST_ADD(4, clock64() - st_p); ST_ADD(5, 1); }
#endif
        if (mode == 2) {
            const double plr = lr_now(gt_prior(prevFreq, e.somatic));
            if (plr > lr_conv) { len = prevLen; freq = prevFreq; shift = 0; }
            else { x0 = s_slot[tid]; E0 = s_slot[T + tid]; E1 = s_slot[2 * T + tid]; E2 = s_slot[3 * T + tid]; }
            break;
        }
        if (mode == 0) {
            s_slot[tid] = x0; s_slot[T + tid] = E0; s_slot[2 * T + tid] = E1; s_slot[3 * T + tid] = E2;     // own entries only: no barrier
            __syncthreads();                              // sh.rgw / sh.nvisited visible
        }
        else {
            double fs = 0, dummy = 0;
            if (has && sub == 0) { const double p0 = E0 * gt.a, p1 = E1 * gt.b, p2 = E2 * gt.c; fs = (p1 + 2 * p2) / (p0 + p1 + p2); }
            block_sum2(fs, dummy, sh.red, par);           // update_allele_frequency :467-485 (priors of the previous iteration)
            freq = fs / 2.0 / a.N;
            if (freq == 0) break;
            gt = gt_prior(freq, e.somatic);
            bool conv = false;
            for (int i = 0; i < sh.nvisited; ++i)
                if (sh.visited_len[i] == (int)len && fabs(sh.visited_freq[i] - freq) <= 0.0001) conv = true;
            if (conv) {
                // convergence :632-658: compare with the previous estimate evaluated with the initial (zero) shifts
                lr_conv = lr_now(gt);
                mode = 2; dlL = (int)prevLen; dlS = 0;
                continue;
            }
        }
        if (!(len >= e.min_len && it < e.iterations)) break;
        ++it;
        prevLen = len; prevFreq = freq;
        const double r0 = sh.rgw[0], r1 = sh.rgw[1], r2 = sh.rgw[2];
        const double aSumRg = r0 * gt.a + r1 * gt.b + r2 * gt.c;
        const double ea0Rg = r0 * gt.a / aSumRg, ea1Rg = r1 * gt.b / aSumRg;      // NaN when read group 0 is high-coverage
        // update_deletion_length :388-462 from the moments of the posterior weights
        double sumDel = 0, wDel = 0;
        if (usable) {
            const double inv = 1.0 / (E0 * gt.a + E1 * gt.b + E2 * gt.c);
            const double ea1 = E1 * gt.b * inv, ea2 = E2 * gt.c * inv;
            if (sub == 0) { sumDel = ea1 * Sr + ea2 * dn; wDel = ea1 * Srd + ea2 * Sd; }
            const double sumRef = ea1Rg * (dn - Sr) + ea0Rg * dn, wRef = ea1Rg * (Sd - Srd) + ea0Rg * Sd;
            const double q = wRef / sumRef;
            int sft = (q != q) ? 0 : (q >= 2147483647.0 ? INT_MAX : (q <= -2147483648.0 ? INT_MIN : (int)q));
            const double sd = __ldg(&a.rgc[s].stddev);
            if (sft > sd || sft < -1 * sd) sft = 0;
            shift = sft;
        }
        block_sum2(sumDel, wDel, sh.red, par);
        if (tid == 0) {                                   // visited[prevLen] = prevFreq (:600); read after the next barrier
            int f = -1;
            for (int i = 0; i < sh.nvisited; ++i) if (sh.visited_len[i] == (int)prevLen) f = i;
            if (f < 0) { f = sh.nvisited++; sh.visited_len[f] = (int)prevLen; }
            sh.visited_freq[f] = prevFreq;
            if ((int)w == e.dbg_window)
                printf("GPU w %u L0 %d it %u len %u freq %.17g sumDel %.17g wDel %.17g\n", w, L0, it, len, freq, sumDel, wDel);
        }
        if (sumDel == 0) len = 0;
        else { const double nlen = wDel / sumDel; len = nlen < 0 ? 0u : (uint32_t)round(nlen); }
        mode = 1; dlL = (int)len; dlS = shift;
    }
#ifdef PD_EM_STATS
    ST_CLK(20, st_t); st_t = clock64();
    if (tid == 0) ST_ADD(9, it);
#endif
    if (freq < 0.0000000001 || len < e.min_len) {
        if (tid == 0) {
            e.valid[blockIdx.x] = 0; if (e.dbg) { e.dbg[4 * blockIdx.x] = 2; e.dbg[4 * blockIdx.x + 1] = len; e.dbg[4 * blockIdx.x + 2] = it; }
        }
        return;
    }
    // ---- final pass :665-727 (compute_data_likelihoods final overload :255-337)
    auto reject = [&](uint32_t reason) {
        if (tid == 0) {
            e.valid[blockIdx.x] = 0;
            if (e.dbg) { e.dbg[4 * blockIdx.x] = reason; e.dbg[4 * blockIdx.x + 1] = len; e.dbg[4 * blockIdx.x + 2] = it; }
        }
    };
    const int flen = (int)len;
    __syncthreads();                                      // s_slot (read above) shares its memory with s_first / s_last (written below)
    const int lower_q = __ldg(&a.rgc[has ? s : 0].lower_q), upper_q = __ldg(&a.rgc[has ? s : 0].upper_q);
    const int inner_off = __ldg(&a.rgc[has ? s : 0].inner_off);
    const double l10_min_prob = __ldg(&a.rgc[has ? s : 0].l10_min_prob);
    const int delLower = usable ? flen - lower_q : INT_MAX, delUpper = usable ? flen + upper_q : 0;
    const uint32_t * pp = e.pool_pos + poff;
    // the read pairs of a lane in batches of FINAL_BATCH, over the warp's largest count so that the batches stay warp-uniform
    const int nlw = __reduce_max_sync(PD_FULL, nl);
    unsigned long long supp = 0, ndata = 0;
    {
        // The ln sums of the final overload (:255-337) equal those of the likelihood pass the registers hold (same read pairs,
        // length and shift: see the state machine above), so only the log10 sums, LAD / DAD and the positions are taken
        // here, from the second half of the table rows {log10, log10p, val, fr}. A batch issues all its deviation, table
        // and position loads before any value-dependent branch; the log10 sums still add the read pairs of a lane in order.
        // (lad1 and dad4 are what the other classes leave of the lane's nl read pairs: two registers fewer in the loop)
        uint32_t lad0 = 0, lad2 = 0, dad0 = 0, dad1 = 0, dad2 = 0, dad3 = 0, nsp = 0;
        uint32_t fl_min = 0xFFFFFFFFu, fl_max = 0, ndeg = 0;
        double t0 = 0, t1 = 0, t2 = 0;
        const uint32_t lane_lt = (1u << (tid & 31)) - 1u;
        for (int b = 0; b < nlw; b += FINAL_BATCH) {
            int d[FINAL_BATCH]; uint32_t first[FINAL_BATCH]; D4 r2[FINAL_BATCH], d2[FINAL_BATCH];
#pragma unroll
            for (int j = 0; j < FINAL_BATCH; ++j) {
                const int jj = b + j;
                d[j] = jj < nl ? (jj < SLOTS ? cache_dev[jj * T + tid] : __ldg(pd + sub + jj * LPS)) : 0;
                first[j] = jj < nl ? __ldg(pp + sub + jj * LPS) + e.anchor : 0u;
            }
#pragma unroll
            for (int j = 0; j < FINAL_BATCH; ++j) {
                const bool v = b + j < nl;
                const uint32_t ir = tab_in(k, d[j] - shift) ? (uint32_t)(d[j] - shift + k.hist_base + 1) : 0u;
                const uint32_t id = v && tab_in(k, d[j] - flen) ? (uint32_t)(d[j] - flen + k.hist_base + 1) : 0u;
                r2[j] = D4{0, 0, 0, 0};
                if (v) r2[j] = ld4(&k.fl[ir].l10);                                                     // log10 ref, log10p, ref, fr
                d2[j] = D4{l10_min_prob, 0, k.min_prob, 0};                                            // floor: .b / .d unused
                if (id) d2[j] = ld4(&k.fl[id].l10);
            }
            uint32_t mine = 0;                                                         // this lane's supporting read pairs, bit j
#pragma unroll
            for (int j = 0; j < FINAL_BATCH; ++j) {
                const int dj = d[j];
                if (b + j >= nl) continue;
                mine |= (uint32_t)(dj >= delLower && dj <= delUpper) << j;
                if (dj > upper_q) { if (dj < delLower) ++dad2; else if (dj <= delUpper) ++dad3; }
                else { if (dj < delUpper) ++dad0; else ++dad1; }
                const double ref = r2[j].c, del = d2[j].c;
                if (ref >= 2 * del) ++lad0; else if (del >= 2 * ref) ++lad2;
                t0 += r2[j].a; t2 += d2[j].a;
                if (ref == del) { t1 += r2[j].a; ++ndeg; }                              // residue applied below
                else if (del == k.min_prob) t1 += r2[j].b;
                else if (ref == k.min_prob) t1 += d2[j].b;
                else t1 += log10(ref + del) - LOG10_2_D;
                fl_min = min(fl_min, first[j]); fl_max = max(fl_max, first[j] + (uint32_t)max(0, dj + inner_off));
            }
            nsp += __popc(mine);
            const uint32_t nsup = __reduce_add_sync(PD_FULL, __popc(mine));
            if (nsup) {
                // one shared reservation per warp and batch (the entries' order does not matter: the percentiles bisect values)
                uint32_t slot = 0;
                if ((tid & 31) == 0) slot = atomicAdd(&s_nsupp, nsup);
                slot = __shfl_sync(PD_FULL, slot, 0);
#pragma unroll
                for (int j = 0; j < FINAL_BATCH; ++j) {
                    const uint32_t m = __ballot_sync(PD_FULL, (mine >> j) & 1u);
                    if ((mine >> j) & 1u) {
                        const uint32_t at = slot + __popc(m & lane_lt);
                        if (at < SUPP_CAP) { s_first[at] = first[j]; s_last[at] = first[j] + (uint32_t)max(0, d[j] + inner_off); }
                    }
                    slot += __popc(m);
                }
            }
        }
        supp = nsp;
        uint32_t lad1 = (uint32_t)nl - lad0 - lad2, dad4 = (uint32_t)nl - dad0 - dad1 - dad2 - dad3;
        lad0 = group_sum<LPS>(lad0, gmask); lad1 = group_sum<LPS>(lad1, gmask); lad2 = group_sum<LPS>(lad2, gmask);
        dad0 = group_sum<LPS>(dad0, gmask); dad1 = group_sum<LPS>(dad1, gmask); dad2 = group_sum<LPS>(dad2, gmask);
        dad3 = group_sum<LPS>(dad3, gmask); dad4 = group_sum<LPS>(dad4, gmask); ndeg = group_sum<LPS>(ndeg, gmask);
        fl_min = group_min<LPS>(fl_min, gmask); fl_max = group_max<LPS>(fl_max, gmask);
        t0 = group_sum<LPS>(t0, gmask); t1 = group_sum<LPS>(t1, gmask); t2 = group_sum<LPS>(t2, gmask);
        if (fl_min == 0xFFFFFFFFu) fl_min = 0;
        double g0l = t0, g1l = t1, g2l = t2;
        if (t0 + t1 + t2 == 0.0) { x0 = 0; E0 = 1.0; E1 = E2 = exp(LN1E10); }     // sum(gtLogs) == 0 :307-308
        else {
            const double mg = fmax(fmax(t0, t1), t2);
            g0l -= mg; g1l -= mg; g2l -= mg;
            if (ndeg) { g1l += ndeg * LOG10_2_RESIDUE; const double m2 = fmax(fmax(g0l, g1l), g2l); g0l -= m2; g1l -= m2; g2l -= m2; }
            if (g0l == g1l && g0l == g2l) { g0l = 0; g1l = -10; g2l = -10; }
        }
        if (has && sub == 0) {
            // calculatePhredGL utils_popdel.h:1511-1528
            const double gTot = log10(exp(g0l) + exp(g1l) + exp(g2l));
            const double q0 = -10 * (g0l - gTot), q1 = -10 * (g1l - gTot), q2 = -10 * (g2l - gTot);
            const double mn = fmin(fmin(q0, q1), q2);
            uint32_t * o = e.ps + (size_t)blockIdx.x * 13 * a.N + 13 * s;
            const bool low = e.sstat[(size_t)job * a.N + s] == 0;
            o[0] = low ? 0u : (uint32_t)round(q0 - mn);
            o[1] = low ? 0u : (uint32_t)round(q1 - mn);
            o[2] = low ? 0u : (uint32_t)round(q2 - mn);
            o[3] = lad0; o[4] = lad1; o[5] = lad2;
            o[6] = dad0; o[7] = dad1; o[8] = dad2; o[9] = dad3; o[10] = dad4;
            o[11] = fl_min; o[12] = fl_max;
            if (!low) ++ndata;
        }
    }
    __syncthreads();
#ifdef PD_EM_STATS
    ST_CLK(6, st_t); st_t = clock64();
    if (tid == 0) ST_ADD(13, 1);
#endif
    block_sum2u(supp, ndata, sh.redu);
    if (supp == 0) { reject(3); return; }
    // percentiles of the supporting starts (80th) and ends (20th): getSuppFirstLast :514-529, by value bisection
    const unsigned long long kF = (unsigned long long)round((double)(supp - 1) * 0.8);
    const unsigned long long kL = (unsigned long long)round((double)(supp - 1) * (1 - 0.8));
    uint32_t sF, sL;
    if (supp <= SUPP_CAP) {
        // start percentile on warp 0, end percentile on warp 1 (both on warp 0 in a one-warp block)
        const uint32_t ns = (uint32_t)supp;
        for (int q = tid >> 5; q < 2; q += T >> 5) {
            const uint32_t * v = q == 0 ? s_first : s_last;
            const unsigned long long kq = q == 0 ? kF : kL;
            uint32_t lo = 0xFFFFFFFFu, hi = 0;
            for (uint32_t i = tid & 31; i < ns; i += 32) { lo = min(lo, v[i]); hi = max(hi, v[i]); }
            lo = __reduce_min_sync(PD_FULL, lo); hi = __reduce_max_sync(PD_FULL, hi);
            while (lo < hi) {
                const uint32_t mid = lo + (hi - lo) / 2;
                uint32_t c = 0;
                for (uint32_t i = tid & 31; i < ns; i += 32) c += v[i] <= mid;
                if (__reduce_add_sync(PD_FULL, c) >= kq + 1) hi = mid; else lo = mid + 1;
            }
            if ((tid & 31) == 0) sh.sel[q] = lo;
        }
        __syncthreads();
        sF = sh.sel[0]; sL = sh.sel[1];
    } else {                                              // more supporting read pairs than the shared list holds: recount per step
        uint32_t loF = 0, hiF = 0xFFFFFFFFu, loL = 0, hiL = 0xFFFFFFFFu;
        while (loF < hiF || loL < hiL) {
            const uint32_t midF = loF + (hiF - loF) / 2, midL = loL + (hiL - loL) / 2;
            unsigned long long cF = 0, cL = 0;
            for (int b = 0; b < nl; b += FINAL_BATCH) {
                int d[FINAL_BATCH]; uint32_t first[FINAL_BATCH];
#pragma unroll
                for (int j = 0; j < FINAL_BATCH; ++j) {
                    const int jj = b + j;
                    d[j] = jj < nl ? (jj < SLOTS ? cache_dev[jj * T + tid] : __ldg(pd + sub + jj * LPS)) : 0;
                    first[j] = jj < nl ? __ldg(pp + sub + jj * LPS) + e.anchor : 0u;
                }
#pragma unroll
                for (int j = 0; j < FINAL_BATCH; ++j) {
                    if (b + j < nl && d[j] >= delLower && d[j] <= delUpper) {
                        const uint32_t last = first[j] + (uint32_t)max(0, d[j] + inner_off);
                        cF += first[j] <= midF; cL += last <= midL;
                    }
                }
            }
            block_sum2u(cF, cL, sh.redu);
            if (loF < hiF) { if (cF >= kF + 1) hiF = midF; else loF = midF + 1; }
            if (loL < hiL) { if (cL >= kL + 1) hiL = midL; else loL = midL + 1; }
        }
        sF = loF; sL = loL;
    }
#ifdef PD_EM_STATS
    ST_CLK(7, st_t); st_t = clock64();
    if (tid == 0) ST_ADD(21, supp);
#endif
    if (sF == 0 && sL == 0) { reject(4); return; }
    const double lr = lr_now(gt);
#ifdef PD_EM_STATS
    ST_CLK(1, st_begin);
#endif
    if (tid == 0) {
        const bool ok = lr >= e.min_lr;
        e.valid[blockIdx.x] = ok ? 1 : 0;
        if (e.dbg) { e.dbg[4 * blockIdx.x] = ok ? 0 : 5; e.dbg[4 * blockIdx.x + 1] = len; e.dbg[4 * blockIdx.x + 2] = it; e.dbg[4 * blockIdx.x + 3] = (uint32_t)supp; }
        if (ok) {
            pd_call c;
            c.initial_length = (uint32_t)L0; c.iterations = it; c.deletion_length = len;
            c.filter = ((double)ndata / a.N >= e.min_sample_fraction) ? 0u : 4u;
            c.lr = lr; c.frequency = freq;
            const uint32_t cur = e.anchor + w * PD_WIN;
            c.window_position = cur - 1;
            c.position = e.window_wise ? cur - 1 : sF;
            c.end_position = e.window_wise ? 0u : sL;
            c.segment = (uint32_t)(((uint64_t)w * PD_WIN) / a.window_buffer);
            e.calls[blockIdx.x] = c;
        }
    }
}

template <int LPS, int SLOTS, int BATCH, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB) k_em_one(PdDev a, EmArgs e)
{
    __shared__ EmShared sh;
    __shared__ __align__(16) uint32_t s_sup[2 * SUPP_CAP];
    uint32_t * s_first = s_sup, * s_last = s_sup + SUPP_CAP;
    __shared__ uint32_t s_nsupp;
    __shared__ uint16_t s_perm[256];
    extern __shared__ int32_t cache_dev[];              // [SLOTS][T] deviations of this block's read pairs
    // parked likelihood triples (first pass / state before the convergence check): only live during the EM loop, so they
    // share the memory of the supporting read-pair lists of the final pass
    static_assert(4 * MAXT * sizeof(double) <= 2 * SUPP_CAP * sizeof(uint32_t), "s_slot must fit the supporting lists");
    double * s_slot = reinterpret_cast<double *>(s_sup);
    em_one_body<LPS, SLOTS, BATCH>(a, e, sh, s_first, s_last, s_nsupp, s_perm, cache_dev, s_slot);
    publish_done(e, blockIdx.x);
}
// ------------------------------------------------------------------------------------------------------------------
// emission: calls of a chunk in pair order -> mapped host memory
// ------------------------------------------------------------------------------------------------------------------
// One kernel per EM chunk on the second stream, CONCURRENT with the chunk's EM launch: a few blocks walk the pairs in
// order in batches of one pair per warp, wait until every pair up to the end of their batch has published `done`
// (acquire), number the valid pairs in pair order (= the reference's call order) and copy call header + per-sample
// row into mapped host memory over PCIe while the EM of later pairs is still running. The last block to finish
// advances the call counter for the next chunk.
constexpr int EMIT_BLOCKS = 12, EMIT_WARPS = 16;

__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t * p)
{
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__global__ void __launch_bounds__(EMIT_WARPS * 32) k_emit_stream(EmitArgs m)
{
    __shared__ uint32_t s_cnt[EMIT_WARPS];
    __shared__ uint32_t s_last;
    const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint32_t base0 = m.counters[CNT_CALLS];            // calls emitted by the earlier chunks (advanced by the LAST block only)
    uint32_t ready = 0, counted = 0, below = 0;              // pairs known done / pairs counted / valid pairs among the counted
    for (uint32_t lo = blockIdx.x * EMIT_WARPS; lo < m.npairs; lo += gridDim.x * EMIT_WARPS) {
        const uint32_t hi = min(lo + (uint32_t)EMIT_WARPS, m.npairs);
        // ---- wait until pairs [0, hi) are final
        const long long t0 = clock64();
        for (;;) {
            bool ok = true;
            for (uint32_t i = ready + tid; i < hi; i += blockDim.x) ok = ok && ld_acquire_gpu(m.done + i) != 0;
            if (__syncthreads_and(ok)) break;
            const bool bad = *(volatile uint32_t *)(m.counters + CNT_ERR) != 0 || clock64() - t0 > 20000000000ll;     // ~10 s: EM kernel gone
            if (__syncthreads_or(bad)) { if (tid == 0) atomicExch(m.counters + CNT_ERR, 1u); return; }
            __nanosleep(200);
        }
        ready = hi;
        // ---- valid pairs below the batch
        uint32_t c = 0;
        for (uint32_t i = counted + tid; i < lo; i += blockDim.x) c += m.valid[i] != 0;
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(PD_FULL, c, o);
        __syncthreads();
        if (lane == 0) s_cnt[wid] = c;
        __syncthreads();
        for (int w = 0; w < EMIT_WARPS; ++w) below += s_cnt[w];
        counted = lo;
        // ---- one warp per pair of the batch
        const uint32_t b = lo + wid;
        uint32_t before = 0;
        for (uint32_t i = lo; i < min(b, hi); ++i) before += m.valid[i] != 0;
        if (b < hi && m.valid[b]) {
            const size_t slot = (size_t)base0 + below + before;
            if (lane == 0) m.out_calls[slot] = m.calls[b];
            const uint4 * src = reinterpret_cast<const uint4 *>(m.ps + (size_t)b * m.row_words);
            uint32_t * dst = m.out_ps + slot * m.row_words;
            const uint32_t n4 = ((size_t)b * m.row_words % 4 == 0 && (slot * m.row_words) % 4 == 0) ? m.row_words / 4 : 0;
            for (uint32_t i = lane; i < n4; i += 32) reinterpret_cast<uint4 *>(dst)[i] = src[i];
            for (uint32_t i = n4 * 4 + lane; i < m.row_words; i += 32) dst[i] = m.ps[(size_t)b * m.row_words + i];
        }
    }
    // ---- the last block to finish publishes the new total (every block has read base0 by then)
    __syncthreads();
    if (tid == 0) { __threadfence(); s_last = atomicAdd(m.emit_blocks_done, 1u) == gridDim.x - 1; }
    __syncthreads();
    if (!s_last) return;
    uint32_t c = 0;
    for (uint32_t i = tid; i < m.npairs; i += blockDim.x) c += m.valid[i] != 0;
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(PD_FULL, c, o);
    if (lane == 0) s_cnt[wid] = c;
    __syncthreads();
    if (tid == 0) {
        uint32_t tot = 0;
        for (int w = 0; w < EMIT_WARPS; ++w) tot += s_cnt[w];
        m.counters[CNT_CALLS] = base0 + tot;
        *m.out_count = base0 + tot;
        *m.emit_blocks_done = 0;
    }
}

template <int LPS, int SLOTS, int MAXT, int MINB>
cudaError_t launch_em_t(const PdDev & a, const EmArgs & e, uint32_t T, cudaStream_t st)
{
    const size_t smem = (size_t)SLOTS * T * (sizeof(double) + sizeof(int32_t));
    cudaError_t err = cudaFuncSetAttribute(k_em<LPS, SLOTS, MAXT, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    k_em<LPS, SLOTS, MAXT, MINB><<<e.npairs, T, smem, st>>>(a, e);
    k_final<LPS, MAXT, MINB><<<e.npairs, T, 0, st>>>(a, e);
    return cudaGetLastError();
}

template <int LPS, int SLOTS, int MAXT, int MINB>
cudaError_t launch_xr_t(const PdDev & a, const EmArgs & e, uint32_t T, cudaStream_t st)
{
    const size_t smem = (size_t)SLOTS * T * (sizeof(double) + sizeof(int32_t));
    cudaError_t err = cudaFuncSetAttribute(k_em_xr<LPS, SLOTS, MAXT, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    err = cudaMemsetAsync(e.xr.ticket, 0, 8, st);
    if (err != cudaSuccess) return err;
    const uint32_t grid = std::max<uint32_t>(1, std::min<uint32_t>(e.npairs, e.xr.grid_cap));
    EmArgs e2 = e;
    e2.xr.epoch = 2 * e.xr.epoch;
    k_em_xr<LPS, SLOTS, MAXT, MINB><<<grid, T, smem, st>>>(a, e2);
    e2.xr.epoch = 2 * e.xr.epoch + 1;
    k_final_xr<LPS, MAXT, MINB><<<grid, T, 0, st>>>(a, e2);
    return cudaGetLastError();
}

template <int LPS, int SLOTS, int MAXT, int MINB, int BATCH>
cudaError_t launch_one_t(const PdDev & a, const EmArgs & e, uint32_t T, cudaStream_t st)
{
    const size_t smem = (size_t)SLOTS * T * sizeof(int32_t);
    k_em_one<LPS, SLOTS, BATCH, MAXT, MINB><<<e.npairs, T, smem, st>>>(a, e);
    return cudaGetLastError();
}

}  // namespace

#ifdef PD_EM_STATS
extern "C" int pd_debug_em_stats(unsigned long long * out)
{
    unsigned long long z[32] = {};
    if (cudaMemcpyFromSymbol(out, g_em_stats, sizeof(z)) != cudaSuccess) return -1;
    if (cudaMemcpyToSymbol(g_em_stats, z, sizeof(z)) != cudaSuccess) return -1;
    return 0;
}
#endif

// CUDA loads kernels lazily, and loading may wait for running kernels: a sharded rank whose first k_final_xr launch had
// to load the kernel while its k_em_xr blocks spin on a peer (whose launch sits behind the same lock) would never
// return. Load the cross-rank kernels up front (pd_shard_attach_*).
int pd_em_preload_xr(pd_ctx * c)
{
    cudaFuncAttributes fa;
    PD_CUDA(c, cudaFuncGetAttributes(&fa, k_em_xr<4, 8, 512, 2>));
    PD_CUDA(c, cudaFuncGetAttributes(&fa, k_em_xr<2, 16, 512, 2>));
    PD_CUDA(c, cudaFuncGetAttributes(&fa, k_final_xr<4, 512, 2>));
    PD_CUDA(c, cudaFuncGetAttributes(&fa, k_final_xr<2, 512, 2>));
    PD_CUDA(c, cudaFuncGetAttributes(&fa, k_emit_stream));
    return 0;
}

int pd_launch_em(pd_ctx * c, const PdDev & a, const EmArgs & e, cudaStream_t st, uint64_t * launches)
{
    if (e.xr.world > 1) {
        // sample-sharded cohort: general kernels with in-kernel cross-rank reductions, persistent blocks (2 per SM at most)
        const uint32_t lpsx = a.N <= 112 ? 4 : (a.N <= 224 ? 2 : 4);
        const uint32_t Tx = std::min<uint32_t>(512, ((a.N * lpsx + 31) / 32) * 32);
        const cudaError_t errx = lpsx == 4 ? launch_xr_t<4, 8, 512, 2>(a, e, Tx, st) : launch_xr_t<2, 16, 512, 2>(a, e, Tx, st);
        if (errx != cudaSuccess) return pd_fail(c, PD_ERR_CUDA, std::string("k_em_xr/k_final_xr launch: ") + cudaGetErrorString(errx));
        *launches += 2;
        return 0;
    }
    // one read group per sample and the cohort fits one block: fused EM + final pass with per-sample state in registers.
    // Measured on B200 (100 samples x chr21, ms per step): one look-up pair in flight at 80 registers / 6 blocks per SM
    // 3.44; two in flight at 96 registers / 5 blocks 3.56; 3 / 4 in flight 3.72 / 4.02; 72 / 64 registers (7 / 8 blocks,
    // spills) 3.78 / 3.86; L1 prefetch of the table rows 5.0; two lanes per sample 5.4; EM loop and final pass as two
    // kernels 3.56-3.76. Final pass, A/B on one B200 at 1000 W, all at 80 registers / 6 blocks: one read pair per
    // iteration with a shared atomic per supporting pair 3.79; FINAL_BATCH = 2 read pairs per lane in flight with one
    // reservation per warp and batch 3.68; 4 in flight 4.07 (spills inside the loop).
    if (a.R == a.N && a.N <= 256 && !getenv("PD_EM_GENERAL")) {
        const uint32_t T1 = ((a.N + 31) / 32) * 32;
        const cudaError_t err1 = T1 <= 128 ? launch_one_t<1, 32, 128, 6, 1>(a, e, T1, st) : launch_one_t<1, 32, 256, 3, 2>(a, e, T1, st);
        if (err1 != cudaSuccess) return pd_fail(c, PD_ERR_CUDA, std::string("k_em_one launch: ") + cudaGetErrorString(err1));
        *launches += 1;
        return 0;
    }
    // lanes per sample (LPS): small cohorts get several lanes per sample so that one block covers all samples at once;
    // each (LPS, block size) class has its own register budget (launch bounds) to keep >= 2 blocks per SM
    const uint32_t N = a.N;
    uint32_t lps = N <= 112 ? 4 : (N <= 224 ? 2 : 4);
    if (getenv("PD_EM_LPS")) lps = (uint32_t)atoi(getenv("PD_EM_LPS"));           // tuning knob
    const uint32_t T = std::min<uint32_t>(512, ((N * lps + 31) / 32) * 32);
    cudaError_t err;
    if (lps == 4) err = T <= 448 ? launch_em_t<4, 8, 448, 2>(a, e, T, st) : launch_em_t<4, 8, 512, 2>(a, e, T, st);
    else if (lps == 2) err = T <= 224 ? launch_em_t<2, 16, 224, 4>(a, e, T, st) : launch_em_t<2, 16, 512, 2>(a, e, T, st);
    else if (lps == 1) err = T <= 128 ? launch_em_t<1, 32, 128, 4>(a, e, T, st) : launch_em_t<1, 32, 512, 2>(a, e, T, st);
    else if (lps == 8) err = launch_em_t<8, 6, 512, 2>(a, e, T, st);
    else return pd_fail(c, PD_ERR_ARG, "PD_EM_LPS must be 1, 2, 4 or 8");
    if (err != cudaSuccess) return pd_fail(c, PD_ERR_CUDA, std::string("k_em/k_final launch: ") + cudaGetErrorString(err));
    *launches += 2;
    return 0;
}

void pd_launch_emit(const EmitArgs & m, cudaStream_t st, uint64_t * launches)
{
    const uint32_t grid = std::max<uint32_t>(1, std::min<uint32_t>(EMIT_BLOCKS, (m.npairs + EMIT_WARPS - 1) / EMIT_WARPS));
    k_emit_stream<<<grid, EMIT_WARPS * 32, 0, st>>>(m);
    ++*launches;
}
