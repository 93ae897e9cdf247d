// pd_host.cu -- host side of the scan library: context, histogram preprocessing, the push path with the
// active-coverage cap, packing into the tiled 32-bit layout, upload, and the host-only validation hook.
#include <mutex>
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <functional>
#include <queue>
#include <string>
#include <vector>

#include "pd_context.h"

static std::string g_create_error;
static void free_words(pd_ctx * c, PdHostRg & h);

// (pd_contig_push may run concurrently for different read groups of one context: the first error wins, under a lock)
int pd_fail(pd_ctx * c, int status, const std::string & msg)
{
    static std::mutex mu;
    if (c) {
        std::lock_guard<std::mutex> lk(mu);
        if (c->status == 0) { c->err = msg; c->status = status; }
    }
    return status;
}

#define PD_CUDA(c, call)                                                                          \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess)                                                                    \
            return pd_fail((c), PD_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

// ---------------------------------------------------------------------------------------------------------
// processHistogram (reference insert_histogram_popdel.h:974-986): smoothing :759-778, quantile distances
// :609-646, density scaling :884-891, per-window normalisation :718-745, probability floor :793-808.
// The reference's integer-accumulator and off-by-one behaviour is part of the contract (SURVEY.md App. C-6).
// ---------------------------------------------------------------------------------------------------------
extern "C" double pd_process_histogram(double * values, uint32_t len, int32_t offset, uint32_t median,
                                       uint32_t read_length, int smoothing, uint32_t pseudo_count_fraction,
                                       uint32_t * lower_q, uint32_t * upper_q)
{
    const int n = (int)len;
    std::vector<double> v(values, values + len);
    if (smoothing) {
        double kern[41], ksum = 0;
        for (int j = -20; j <= 20; ++j) { kern[j + 20] = std::exp(-j * j / 40.0); }
        for (int j = 0; j < 41; ++j) ksum += kern[j];             // all 41 weights, also outside the histogram
        std::vector<double> sm(len);
        for (int i = 0; i < n; ++i) {
            double acc = 0;
            for (int j = -20; j <= 20; ++j)
                if (i + j >= 0 && i + j < n) acc += kern[j + 20] * v[i + j];
            sm[i] = acc / ksum;
        }
        v.swap(sm);
    }
    uint32_t lq = 0, uq = 0;
    {
        unsigned total = 0;                                       // `unsigned += double`: truncates each step
        for (int i = 1; i + 1 < n; ++i) total += v[i];
        const double lower = total * 0.01, upper = total * 0.99;
        double run = 0;
        int i = 1;
        for (; i + 1 < n; ++i) {
            run += v[i];
            if (run >= lower) { lq = (uint32_t)std::abs(i + offset - (int)median); break; }
        }
        for (; i + 1 < n; ++i) {                                  // restarts on the same element: counted twice
            run += v[i];
            if (run >= upper) { uq = (uint32_t)std::abs(i + offset - (int)median); break; }
        }
    }
    {
        unsigned total = 0;
        for (int i = 0; i < n; ++i) total += v[i];
        for (int i = 0; i < n; ++i) v[i] /= total;
    }
    {
        unsigned isize = (unsigned)offset;                        // index 1 is paired with insert size `offset`
        for (int i = 1; i + 1 < n; ++i, ++isize) {
            int inner = (int)(isize - 2 * read_length);
            if (inner < 1) inner = 1;
            v[i] *= static_cast<double>(256 + inner - 1) / 256;
        }
    }
    double mx = 0;
    for (int i = 0; i < n; ++i) mx = std::max(mx, v[i]);
    const double min_prob = mx / pseudo_count_fraction;
    for (int i = 0; i < n; ++i) values[i] = v[i] < min_prob ? min_prob : v[i];
    if (lower_q) *lower_q = lq;
    if (upper_q) *upper_q = uq;
    return min_prob;
}

// ---------------------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------------------
extern "C" const char * pd_create_error(void) { return g_create_error.c_str(); }
extern "C" const char * pd_last_error(pd_ctx * c) { return c ? c->err.c_str() : "null context"; }

static int upload_static(pd_ctx * c)
{
    // the reference evaluates log(2.0) / log10(2.0) in double (genotype_deletion_popdel_call.h:212,298)
    const double LN2_D = std::log(2.0), L10_2_D = std::log10(2.0);
    size_t total = 0;
    for (auto & t : c->tables_) total += t.size() + 1;
    std::vector<PdTab> tab(total);
    for (uint32_t g = 0; g < c->R; ++g) {
        const double mp = c->rgc[g].min_prob;
        auto fill = [&](PdTab & e, double v) {
            e.val = v; e.ln = std::log(v); e.l10 = std::log10(v);
            e.lnp = std::log(v + mp) - LN2_D; e.l10p = std::log10(v + mp) - L10_2_D;
            e.fr = mp / (mp + v); e.val2 = v; e.fr2 = e.fr;
        };
        size_t o = c->rgc[g].hist_off;
        fill(tab[o], mp);                                           // floor entry
        for (size_t i = 0; i < c->tables_[g].size(); ++i) fill(tab[o + 1 + i], c->tables_[g][i]);
    }
    PD_CUDA(c, cudaMalloc(&c->d_tab, std::max<size_t>(total, 1) * sizeof(PdTab)));
    PD_CUDA(c, cudaMemcpy(c->d_tab, tab.data(), total * sizeof(PdTab), cudaMemcpyHostToDevice));
    PD_CUDA(c, cudaMalloc(&c->d_rgc, c->R * sizeof(PdRgConst)));
    PD_CUDA(c, cudaMemcpy(c->d_rgc, c->rgc.data(), c->R * sizeof(PdRgConst), cudaMemcpyHostToDevice));
    {
        std::vector<uint32_t> mi(c->R);
        for (uint32_t g = 0; g < c->R; ++g) mi[g] = c->rgc[g].min_init;
        PD_CUDA(c, cudaMalloc(&c->d_min_init, c->R * 4));
        PD_CUDA(c, cudaMemcpy(c->d_min_init, mi.data(), c->R * 4, cudaMemcpyHostToDevice));
    }
    PD_CUDA(c, cudaMalloc(&c->d_sample_rg, (c->N + 1) * 4));
    PD_CUDA(c, cudaMemcpy(c->d_sample_rg, c->sample_rg.data(), (c->N + 1) * 4, cudaMemcpyHostToDevice));
    return 0;
}

// stream2 carries the result emitter, which runs concurrently with the EM kernels: its few blocks should get an SM as
// soon as one has room
static cudaError_t create_priority_stream(cudaStream_t * s)
{
    int lo = 0, hi = 0;
    cudaError_t e = cudaDeviceGetStreamPriorityRange(&lo, &hi);
    if (e != cudaSuccess) return e;
    return cudaStreamCreateWithPriority(s, cudaStreamNonBlocking, hi);
}

extern "C" pd_ctx * pd_create(const pd_params * p, uint32_t n_samples, uint32_t n_rg, const pd_rg * rgs, int device)
{
    g_create_error.clear();
    if (!p || !rgs || n_samples == 0 || n_rg < n_samples) { g_create_error = "pd_create: invalid arguments"; return nullptr; }
    if (p->window_size != 30) { g_create_error = "pd_create: only 30-bp windows are supported"; return nullptr; }
    if (p->window_buffer < 960 || p->iterations > 60) { g_create_error = "pd_create: window_buffer < 960 or iterations > 60"; return nullptr; }
    pd_ctx * c = new pd_ctx();
    c->params = *p; c->N = n_samples; c->R = n_rg; c->device = device;
    c->grid.window_buffer = p->window_buffer;
    c->rgs.assign(rgs, rgs + n_rg);
    c->tables_.resize(n_rg);
    c->rgc.resize(n_rg);
    c->sample_rg.assign(n_samples + 1, 0);
    uint32_t hist_off = 0, prev_sample = 0;
    int64_t tmin = INT32_MAX;
    for (uint32_t g = 0; g < n_rg; ++g) {
        const pd_rg & r = rgs[g];
        if (r.sample >= n_samples || r.sample < prev_sample || (g == 0 && r.sample != 0) || r.sample > prev_sample + 1 ||
            !r.values || r.len < 3) {
            g_create_error = "pd_create: read groups must be grouped by sample in ascending order, every sample non-empty";
            delete c; return nullptr;
        }
        prev_sample = r.sample;
        c->sample_rg[r.sample + 1] = g + 1;
        c->tables_[g].assign(r.values, r.values + r.len);
        c->rgs[g].values = c->tables_[g].data();
        PdRgConst & k = c->rgc[g];
        k.inner_off = (int32_t)r.median - 2 * (int32_t)r.read_length;
        k.max_load = r.max_load; k.sample = r.sample; k.median = (int32_t)r.median;
        k.hist_base = (int32_t)r.median - r.offset; k.hist_len = r.len; k.hist_off = hist_off;
        k.min_prob = r.min_prob; k.ln_min_prob = std::log(r.min_prob); k.l10_min_prob = std::log10(r.min_prob);
        k.stddev = r.stddev; k.lower_q = (int32_t)r.lower_quantile_dist; k.upper_q = (int32_t)r.upper_quantile_dist;
        k.min_init = r.min_init_del_len; k.pad_ = 0;
        // stream read pairs with dev up to ~8 sigma stay "short": span <= lookback tiles
        double span_w = (29.0 + std::max(0.0, k.inner_off + 8.0 * r.stddev)) / 30.0 + 2.0;
        uint32_t lb = (uint32_t)std::ceil(span_w / PD_TILE_WINDOWS);
        k.lookback_tiles = std::min<uint32_t>(std::max<uint32_t>(lb, 1), PD_MAX_LOOKBACK_TILES);
        hist_off += r.len + 1;
        tmin = std::min<int64_t>(tmin, r.min_init_del_len);
    }
    if (c->sample_rg[n_samples] != n_rg || prev_sample != n_samples - 1) {
        g_create_error = "pd_create: every sample needs at least one read group"; delete c; return nullptr;
    }
    c->t_min = (int32_t)std::min<int64_t>(tmin, PD_DEV_MAX - 1);
    c->hrg.resize(n_rg);
    c->raw.resize(n_rg);
    if (device >= 0) {
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || device >= ndev) {
            g_create_error = std::string("pd_create: no usable CUDA device (") + (e != cudaSuccess ? cudaGetErrorString(e) : "index out of range") +
                             "); this library has no CPU scan path";
            delete c; return nullptr;
        }
        if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
            create_priority_stream(&c->stream2) != cudaSuccess) {
            g_create_error = "pd_create: cudaSetDevice/cudaStreamCreate failed"; delete c; return nullptr;
        }
        for (auto & ev : c->ev) cudaEventCreate(&ev);
        if (upload_static(c) != 0) { g_create_error = c->err; pd_destroy(c); return nullptr; }
    }
    return c;
}

extern "C" int pd_device_warmup(int device)
{
    if (cudaSetDevice(device) != cudaSuccess || cudaFree(nullptr) != cudaSuccess) { cudaGetLastError(); return PD_ERR_CUDA; }
    return 0;
}

extern "C" void pd_destroy(pd_ctx * c)
{
    if (!c) return;
    if (c->device >= 0) {
        cudaSetDevice(c->device);
        cudaFree(c->d_words); cudaFree(c->d_tiles); cudaFree(c->d_longs);
        pd_shard_release(c);
        pd_unify_release(c);
        for (auto & e : c->ev_pack) if (e) cudaEventDestroy(e);
        cudaFree(c->d_rgc); cudaFree(c->d_sample_rg); cudaFree(c->d_tab); cudaFree(c->d_min_init);
        if (c->res_ps) cudaFreeHost(c->res_ps);
        if (c->res_calls) cudaFreeHost(c->res_calls);
        if (c->res_count) cudaFreeHost(c->res_count);
        cudaFree(c->d_gran_off); cudaFree(c->d_gran_tile); cudaFree(c->d_long_off); cudaFree(c->d_tseg);
        for (auto & p : c->d_scratch) cudaFree(p);
        for (auto & p : c->d_pack) cudaFree(p);
        for (auto & ev : c->ev) if (ev) cudaEventDestroy(ev);
        if (c->stream) cudaStreamDestroy(c->stream);
        if (c->stream2) cudaStreamDestroy(c->stream2);
    }
    for (auto & h : c->hrg) free_words(c, h);
    delete c;
}

// ---------------------------------------------------------------------------------------------------------
// contig: begin / push (active-coverage cap + packing in one pass) / finalise / upload
// ---------------------------------------------------------------------------------------------------------
static void free_words(pd_ctx * c, PdHostRg & h)
{
    if (h.words) { if (h.words_pinned) cudaFreeHost(h.words); else free(h.words); }
    h.words = nullptr; h.n_words = h.cap_words = 0;
}

static bool reserve_words(pd_ctx * c, PdHostRg & h, size_t need)
{
    if (need <= h.cap_words) return true;
    size_t want = std::max<size_t>(need + need / 4, 4096);
    uint32_t * p = nullptr;
    const bool pin = c->device >= 0 && c->pinned_staging;
    if (pin) { if (cudaMallocHost(&p, want * 4) != cudaSuccess) return false; }
    else { p = (uint32_t *)malloc(want * 4); if (!p) return false; }
    if (h.n_words) memcpy(p, h.words, h.n_words * 4);
    uint32_t * old = h.words;
    const bool old_pinned = h.words_pinned;
    h.words = p; h.cap_words = want; h.words_pinned = pin;
    if (old) { if (old_pinned) cudaFreeHost(old); else free(old); }
    return true;
}

extern "C" int pd_contig_begin(pd_ctx * c, uint32_t anchor)
{
    if (!c) return PD_ERR_ARG;
    if (c->status) return c->status;
    if (anchor % PD_WIN != 0) return pd_fail(c, PD_ERR_ARG, "pd_contig_begin: anchor must be a multiple of 30 (first 30-bp window of the contig)");
    c->grid.anchor = anchor;
    for (auto & h : c->hrg) {
        uint32_t * w = h.words; size_t cap = h.cap_words;      // keep the staging buffer across contigs
        const bool pinned = h.words_pinned;
        h = PdHostRg();
        h.words = w; h.cap_words = cap; h.words_pinned = pinned;
        h.tile_rel.assign(1, 0u); h.tile_reach.assign(1, 0xFFFFFFu);
    }
    for (auto & r : c->raw) r = PdRawRg();
    c->dev_mode = c->host_mode = false;
    c->contig_open = true; c->packed = false; c->uploaded = false; c->index_built = false;
    c->n_windows_total = 0; c->n_reads = 0; c->min_windows = 0; c->tail = PdTail();
    return 0;
}

// The cap of ChromosomeProfile::add (profile_structure_popdel_call.h:1084-1113, getEndCount :870-928): a read pair is
// stored while the reference's activeLoad counter of its read group is below max_load (PdCapState, pd_context.h: the
// counter with its lazy refresh at segment switches and the zeroing after a segment without read pairs).
// Thread-compatible: may run concurrently for DIFFERENT read groups of one context.
extern "C" int pd_contig_push(pd_ctx * c, uint32_t rg, uint64_t n, const uint32_t * pos, const int32_t * dev)
{
    if (!c) return PD_ERR_ARG;
    if (c->status) return c->status;
    if (!c->contig_open || rg >= c->R || (n && (!pos || !dev))) return pd_fail(c, PD_ERR_ARG, "pd_contig_push: bad arguments or no open contig");
    if (c->packed) return pd_fail(c, PD_ERR_ARG, "pd_contig_push: contig already packed");
    if (c->dev_mode) return pd_fail(c, PD_ERR_ARG, "pd_contig_push: cannot be mixed with pd_contig_push_pinned in one contig");
    c->host_mode = true;
    PdHostRg & h = c->hrg[rg];
    const PdRgConst & k = c->rgc[rg];
    const bool capped = k.max_load != 0xFFFFFFFFu;
    const uint32_t wb = c->grid.window_buffer, anchor = c->grid.anchor;
    if (!reserve_words(c, h, h.n_words + n + n / 8 + 64)) return pd_fail(c, PD_ERR_CUDA, "pd_contig_push: out of (pinned) host memory");
    uint64_t seg_end_bp = h.seg < 0 ? 0 : (uint64_t)(h.seg + 1) * wb;
    int64_t wl = h.seg < 0 ? -1 : (int64_t)pd_seg_last_window((uint64_t)h.seg, wb);
    int64_t wl2 = h.seg < 0 ? -1 : (int64_t)pd_seg_last_window((uint64_t)h.seg + 1, wb);
    uint32_t * words = h.words;
    size_t nw = h.n_words, cap = h.cap_words;
    const int32_t inner_off = k.inner_off;
    const uint32_t lookback = k.lookback_tiles, max_load = k.max_load;
    PdCapState & cs = h.cap;
    uint32_t cur_tile = h.cur_tile, last_pos = h.last_pos;
    int64_t S = h.S, E_own = h.E_own, E_spill = h.E_spill;
    uint64_t n_reads = h.n_reads, dropped = h.dropped;
    bool any = h.any;
    int rc = 0;
    for (uint64_t i = 0; i < n; ++i) {
        const uint32_t p = pos[i];
        if (p < anchor) { rc = pd_fail(c, PD_ERR_ARG, "pd_contig_push: position before the contig anchor"); break; }
        if (any && p < last_pos) { rc = pd_fail(c, PD_ERR_ORDER, "pd_contig_push: read pairs must be sorted by position"); break; }
        any = true; last_pos = p;
        const uint32_t pr = p - anchor;
        const uint32_t b = pr / PD_WIN, bp = b * PD_WIN;
        const int32_t d = dev[i];
        int64_t inner = (int64_t)d + inner_off;
        if (inner < 0) inner = 0;
        const uint64_t endp = (uint64_t)pr + (uint64_t)inner;
        const int64_t lw = endp < 0xFFFFFFFFull ? (int64_t)((uint32_t)endp / PD_WIN) : (int64_t)(endp / PD_WIN);
        if (capped) {
            if (cs.seg < 0) cs.start(wb);
            if ((uint64_t)bp >= cs.set[cs.write_set].right) {       // every segment switch up to this read pair's segment
                const int64_t j = (int64_t)((uint64_t)bp / wb);
                while (cs.seg < j) cs.next_segment(wb);
            }
            if (!cs.admit(b, (uint32_t)std::min<int64_t>(lw, 0xFFFFFFFF), max_load)) { ++dropped; continue; }
        }
        if (bp >= seg_end_bp || h.seg < 0) {                        // first read pair of a new segment
            const int64_t j = (int64_t)((uint64_t)bp / wb);
            if (h.seg >= 0) { h.prev_seg = h.seg; h.prev_E_spill = E_spill; }
            h.seg = j; S = E_own = E_spill = -1;
            seg_end_bp = (uint64_t)(j + 1) * wb;
            wl = (int64_t)pd_seg_last_window((uint64_t)j, wb);
            wl2 = (int64_t)pd_seg_last_window((uint64_t)j + 1, wb);
        }
        S = pr;                                                     // positions are sorted
        if (lw <= wl) { if (lw > E_own) E_own = lw; } else if (lw > E_spill) E_spill = lw;
        const int64_t s = (int64_t)b + (pr != bp ? 1 : 0);
        int64_t e = lw + 1;
        const bool act = s <= wl;
        if (act) { const int64_t capw = lw <= wl ? wl : wl2; if (e > capw) e = capw; }
        const uint32_t t = b / PD_TILE_WINDOWS;
        if (t != cur_tile) {
            while (nw & 3) words[nw++] = PD_PAD_WORD;
            while (cur_tile < t) { ++cur_tile; h.tile_rel.push_back((uint32_t)nw); h.tile_reach.push_back(0xFFFFFFu); }
        }
        bool is_long = d > PD_DEV_MAX || d < PD_DEV_MIN + 1;
        if (act && (uint64_t)e / PD_TILE_WINDOWS > (uint64_t)t + lookback) is_long = true;
        const int32_t dc = d > PD_DEV_MAX ? PD_DEV_MAX : (d < PD_DEV_MIN + 1 ? PD_DEV_MIN + 1 : d);
        if (nw + 8 > cap) {                                         // padding can outgrow the reservation
            h.n_words = nw;
            if (!reserve_words(c, h, nw + (n - i) + (n - i) / 8 + 64)) { rc = pd_fail(c, PD_ERR_CUDA, "pd_contig_push: out of (pinned) host memory"); break; }
            words = h.words; cap = h.cap_words;
        }
        if (act && !is_long && (uint64_t)e / PD_TILE_WINDOWS > t) {   // PdTile::reach: first word / furthest tile reached by this tile's stream
            uint32_t & tr = h.tile_reach[t];
            const uint32_t far = (uint32_t)std::min<uint64_t>((uint64_t)e / PD_TILE_WINDOWS - t, 255), first = std::min<uint32_t>(tr & 0xFFFFFFu, (uint32_t)(nw - h.tile_rel[t]));
            tr = (std::max(tr >> 24, far) << 24) | std::min(first, 0xFFFFFFu);
        }
        words[nw++] = pd_pack(dc, pr - t * PD_TILE_BP, is_long);
        if (is_long && act) {
            h.longs.push_back(PdLong{(uint32_t)s, (uint32_t)e, pr, d});
            h.long_span = std::max<uint32_t>(h.long_span, (uint32_t)(e - s + 1));
        }
        ++n_reads;
        if (nw > 0xFFFFFFF0ull) { rc = pd_fail(c, PD_ERR_CAPACITY, "more than 2^32 packed words in one read group"); break; }
    }
    h.cur_tile = cur_tile; h.last_pos = last_pos; h.any = any;
    h.S = S; h.E_own = E_own; h.E_spill = E_spill; h.n_reads = n_reads; h.dropped = dropped;
    if (rc) { h.n_words = nw; return rc; }
    h.n_words = nw;
    return 0;
}

// Last window the reference scans for this contig (workflow_popdel.h:42-47 with nextWindow's stop rules,
// profile_structure_popdel_call.h:1213-1247): in the final segment kf the scan runs until the border or until every
// start entry is activated and every end entry of end set kf (own entries ending before the border, spill-over
// entries of segment kf-1) is removed.
uint64_t pd_tail_windows(const PdTail & t, uint32_t wb)
{
    if (t.kf < 0) return 0;
    const int64_t stop = std::max(t.E + 2, (t.S + 29) / (int64_t)PD_WIN);
    const int64_t wl = (int64_t)pd_seg_last_window((uint64_t)t.kf, wb);
    return (uint64_t)std::min(stop, wl) + 1;
}
static uint64_t last_scanned_window(pd_ctx * c)
{
    PdTail t;
    for (const auto & h : c->hrg) t.kf = std::max(t.kf, h.seg);
    if (t.kf >= 0)
        for (const auto & h : c->hrg) {
            if (h.seg == t.kf) {
                t.S = std::max(t.S, h.S); t.E = std::max(t.E, h.E_own); t.E_spill = std::max(t.E_spill, h.E_spill);
                if (h.prev_seg == t.kf - 1) t.E = std::max(t.E, h.prev_E_spill);
            } else if (h.seg == t.kf - 1) t.E = std::max(t.E, h.E_spill);
        }
    c->tail = t;
    return pd_tail_windows(t, c->grid.window_buffer);
}

int pd_pack_contig(pd_ctx * c)
{
    if (c->packed) return 0;
    c->n_windows_total = last_scanned_window(c);
    uint64_t max_tile = (std::max(c->n_windows_total, c->min_windows) + PD_TILE_WINDOWS - 1) / PD_TILE_WINDOWS;
    for (auto & h : c->hrg) {
        if (!reserve_words(c, h, h.n_words + 4)) return pd_fail(c, PD_ERR_CUDA, "out of (pinned) host memory");
        while (h.n_words & 3) h.words[h.n_words++] = PD_PAD_WORD;
        if (h.n_reads) max_tile = std::max<uint64_t>(max_tile, (uint64_t)h.cur_tile + 1);
    }
    if (max_tile + 1 >= (1ull << 31)) return pd_fail(c, PD_ERR_RANGE, "contig too long for the tile index");
    c->NT = (uint32_t)std::max<uint64_t>(max_tile, 1);
    const uint32_t NT = c->NT;
    c->h_tiles.assign((size_t)c->R * (NT + 1), PdTile{0, 0, 0, 0});
    c->h_long_off.assign(c->R + 1, 0);
    c->h_word_base.assign(c->R + 1, 0);
    uint64_t total = 0, nlong = 0;
    c->n_reads = 0;
    for (uint32_t g = 0; g < c->R; ++g) {
        const PdHostRg & h = c->hrg[g];
        c->h_word_base[g] = total;
        if (total + h.n_words > 0xFFFFFFF0ull)
            return pd_fail(c, PD_ERR_CAPACITY, "more than 2^32 packed words in one contig batch; split the cohort or the contig");
        PdTile * tl = &c->h_tiles[(size_t)g * (NT + 1)];
        const size_t seen = h.tile_rel.size();
        // wide-list range per tile: entries are sorted by s; [lo, hi) = first entry still alive (e >= 32t) .. first with s > 32t+31
        size_t lo = 0, hi = 0;
        const size_t nl = h.longs.size();
        for (uint32_t t = 0; t <= NT; ++t) {
            tl[t].off = (uint32_t)(total + (t < seen ? h.tile_rel[t] : h.n_words));
            tl[t].reach = t < h.tile_reach.size() ? h.tile_reach[t] : 0u;
            const uint64_t w0 = (uint64_t)t * PD_TILE_WINDOWS;
            while (hi < nl && h.longs[hi].s <= w0 + PD_TILE_WINDOWS - 1) ++hi;
            while (lo < hi && h.longs[lo].e < w0) ++lo;
            tl[t].long_lo = (uint32_t)(nlong + lo);
            tl[t].long_hi = (uint32_t)(nlong + hi);
        }
        total += h.n_words;
        c->h_long_off[g] = (uint32_t)nlong;
        nlong += nl;
        c->n_reads += h.n_reads;
    }
    c->h_word_base[c->R] = total;
    c->h_long_off[c->R] = (uint32_t)nlong;
    c->total_words = total; c->total_longs = nlong;
    c->packed = true;
    return 0;
}

extern "C" int pd_contig_push_pinned(pd_ctx * c, uint32_t rg, uint64_t n, const uint32_t * pos, const int32_t * dev)
{
    if (!c) return PD_ERR_ARG;
    if (c->status) return c->status;
    if (!c->contig_open || rg >= c->R || (n && (!pos || !dev))) return pd_fail(c, PD_ERR_ARG, "pd_contig_push_pinned: bad arguments or no open contig");
    if (c->device < 0) return pd_fail(c, PD_ERR_CUDA, "pd_contig_push_pinned: host-only context");
    if (c->host_mode || c->packed) return pd_fail(c, PD_ERR_ARG, "pd_contig_push_pinned: cannot be mixed with pd_contig_push / contig already packed");
    if (c->raw[rg].n) return pd_fail(c, PD_ERR_ARG, "pd_contig_push_pinned: one call per read group and contig");
    c->dev_mode = true;
    PdRawRg r; r.pos = pos; r.dev = dev; r.n = n;
    c->raw[rg] = r;
    return 0;
}

extern "C" int pd_contig_push_device(pd_ctx * c, uint32_t rg, uint64_t n, const uint32_t * d_pos, const int32_t * d_dev)
{
    if (!c) return PD_ERR_ARG;
    if (c->status) return c->status;
    if (!c->contig_open || rg >= c->R || (n && (!d_pos || !d_dev))) return pd_fail(c, PD_ERR_ARG, "pd_contig_push_device: bad arguments or no open contig");
    if (c->device < 0) return pd_fail(c, PD_ERR_CUDA, "pd_contig_push_device: host-only context");
    if (c->host_mode || c->packed) return pd_fail(c, PD_ERR_ARG, "pd_contig_push_device: cannot be mixed with pd_contig_push / contig already packed");
    if (c->raw[rg].n) return pd_fail(c, PD_ERR_ARG, "pd_contig_push_device: one call per read group and contig");
    c->dev_mode = true;
    PdRawRg r; r.pos = d_pos; r.dev = d_dev; r.n = n; r.on_device = true;
    c->raw[rg] = r;
    return 0;
}

extern "C" int pd_contig_push_compact32(pd_ctx * c, uint32_t rg, uint64_t n, const uint32_t * words, uint32_t n_blocks, const uint32_t * blk_first)
{
    if (!c) return PD_ERR_ARG;
    if (c->status) return c->status;
    if (!c->contig_open || rg >= c->R || (n && (!words || !blk_first || !n_blocks)) || n_blocks > 0x7FFFFFFFu)
        return pd_fail(c, PD_ERR_ARG, "pd_contig_push_compact32: bad arguments or no open contig");
    if (c->device < 0) return pd_fail(c, PD_ERR_CUDA, "pd_contig_push_compact32: host-only context");
    if (c->host_mode || c->packed) return pd_fail(c, PD_ERR_ARG, "pd_contig_push_compact32: cannot be mixed with pd_contig_push / contig already packed");
    if (c->raw[rg].n) return pd_fail(c, PD_ERR_ARG, "pd_contig_push_compact32: one call per read group and contig");
    if (n && (blk_first[n_blocks] != n || blk_first[0] != 0)) return pd_fail(c, PD_ERR_ARG, "pd_contig_push_compact32: blk_first must run from 0 to n");
    c->dev_mode = true;
    PdRawRg r;
    r.n = n; r.w32 = words; r.blk = blk_first; r.nblk = n_blocks;
    c->raw[rg] = r;
    return 0;
}

extern "C" int pd_contig_push_compact(pd_ctx * c, uint32_t rg, uint64_t n, const uint16_t * pos_lo, const uint8_t * dev24,
                                      uint32_t n_blocks, const uint32_t * blk_first)
{
    if (!c) return PD_ERR_ARG;
    if (c->status) return c->status;
    if (!c->contig_open || rg >= c->R || (n && (!pos_lo || !dev24 || !blk_first || !n_blocks)))
        return pd_fail(c, PD_ERR_ARG, "pd_contig_push_compact: bad arguments or no open contig");
    if (c->device < 0) return pd_fail(c, PD_ERR_CUDA, "pd_contig_push_compact: host-only context");
    if (c->host_mode || c->packed) return pd_fail(c, PD_ERR_ARG, "pd_contig_push_compact: cannot be mixed with pd_contig_push / contig already packed");
    if (c->raw[rg].n) return pd_fail(c, PD_ERR_ARG, "pd_contig_push_compact: one call per read group and contig");
    if (n && (blk_first[n_blocks] != n || blk_first[0] != 0)) return pd_fail(c, PD_ERR_ARG, "pd_contig_push_compact: blk_first must run from 0 to n");
    c->dev_mode = true;
    PdRawRg r;
    r.n = n; r.lo = pos_lo; r.d24 = dev24; r.blk = blk_first; r.nblk = n_blocks;
    c->raw[rg] = r;
    return 0;
}

extern "C" int pd_contig_reserve_windows(pd_ctx * c, uint64_t n_windows)
{
    if (!c) return PD_ERR_ARG;
    if (c->status) return c->status;
    if (!c->contig_open || c->packed || c->uploaded) return pd_fail(c, PD_ERR_ARG, "pd_contig_reserve_windows: call between pd_contig_begin and the upload");
    c->min_windows = n_windows;
    return 0;
}

extern "C" int pd_contig_window_count(pd_ctx * c, uint64_t * n)
{
    if (!c || !n) return PD_ERR_ARG;
    if (c->status) return c->status;
    if (!c->contig_open) return pd_fail(c, PD_ERR_ARG, "no open contig");
    if (c->dev_mode && !c->uploaded) { int rc0 = pd_contig_upload(c); if (rc0) return rc0; }
    if (c->dev_mode) { *n = c->n_windows_total; return 0; }
    int rc = pd_pack_contig(c);
    if (rc) return rc;
    *n = c->n_windows_total;
    return 0;
}

template <typename T>
static int grow(pd_ctx * c, T *& p, size_t & cap, size_t need)
{
    if (need <= cap && p) return 0;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = std::max<size_t>(need + need / 8, 1024);
    PD_CUDA(c, cudaMalloc(&p, want * sizeof(T)));
    cap = want;
    return 0;
}

extern "C" int pd_contig_upload(pd_ctx * c)
{
    if (!c) return PD_ERR_ARG;
    if (c->status) return c->status;
    if (c->device < 0) return pd_fail(c, PD_ERR_CUDA, "pd_contig_upload: host-only context (device = -1); the scan needs a CUDA device");
    if (!c->contig_open) return pd_fail(c, PD_ERR_ARG, "no open contig");
    if (c->uploaded) return 0;
    if (c->dev_mode) {
        int prc = pd_pack_on_device(c);
        if (prc < 0) return prc;
        if (prc == 0) { c->packed = true; c->uploaded = true; c->index_built = false; return 0; }
        // the active-coverage cap would drop read pairs (or a span exceeds the device look-back): sequential host path
        c->dev_mode = false;
        c->raw_pos_dec.assign(c->R, {}); c->raw_dev_dec.assign(c->R, {});
        for (uint32_t g = 0; g < c->R; ++g) {
            PdRawRg r = c->raw[g];
            if (r.on_device && r.n) {                              // device-resident arrays: one copy to the host
                auto & P = c->raw_pos_dec[g]; auto & D = c->raw_dev_dec[g];
                P.resize(r.n); D.resize(r.n);
                PD_CUDA(c, cudaMemcpy(P.data(), r.pos, r.n * 4, cudaMemcpyDeviceToHost));
                PD_CUDA(c, cudaMemcpy(D.data(), r.dev, r.n * 4, cudaMemcpyDeviceToHost));
                r.pos = P.data(); r.dev = D.data();
            }
            if (r.compact() && r.n) {                              // decode the compact arrays for the sequential packer
                auto & P = c->raw_pos_dec[g]; auto & D = c->raw_dev_dec[g];
                P.resize(r.n); D.resize(r.n);
                for (uint32_t b = 0; b < r.nblk && r.w32; ++b)
                    for (uint64_t i = r.blk[b]; i < r.blk[b + 1]; ++i) { P[i] = (b << 8) | (r.w32[i] & 0xFFu); D[i] = (int32_t)r.w32[i] >> 8; }
                for (uint32_t b = 0; b < r.nblk && !r.w32; ++b)
                    for (uint64_t i = r.blk[b]; i < r.blk[b + 1]; ++i) {
                        P[i] = (b << 16) | r.lo[i];
                        const uint32_t u = (uint32_t)r.d24[3 * i] | ((uint32_t)r.d24[3 * i + 1] << 8) | ((uint32_t)r.d24[3 * i + 2] << 16);
                        D[i] = (int32_t)(u << 8) >> 8;
                    }
                r.pos = P.data(); r.dev = D.data();
            }
            int hrc = pd_contig_push(c, g, r.n, r.pos, r.dev);
            if (hrc) return hrc;
        }
        c->raw_pos_dec.clear(); c->raw_dev_dec.clear();
    }
    int rc = pd_pack_contig(c);
    if (rc) return rc;
    PD_CUDA(c, cudaSetDevice(c->device));
    if (grow(c, c->d_words, c->cap_words, c->total_words + 4)) return c->status;
    if (grow(c, c->d_tiles, c->cap_tiles, c->h_tiles.size())) return c->status;
    if (grow(c, c->d_longs, c->cap_longs, c->total_longs + 1)) return c->status;
    PD_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
    c->h2d_bytes = 0;
    for (uint32_t g = 0; g < c->R; ++g) {                         // straight from the pinned per-read-group buffers
        const PdHostRg & h = c->hrg[g];
        if (h.n_words) PD_CUDA(c, cudaMemcpyAsync(c->d_words + c->h_word_base[g], h.words, h.n_words * 4, cudaMemcpyHostToDevice, c->stream));
        if (!h.longs.empty())
            PD_CUDA(c, cudaMemcpyAsync(c->d_longs + c->h_long_off[g], h.longs.data(), h.longs.size() * sizeof(PdLong), cudaMemcpyHostToDevice, c->stream));
        c->h2d_bytes += h.n_words * 4 + h.longs.size() * sizeof(PdLong);
    }
    PD_CUDA(c, cudaMemcpyAsync(c->d_tiles, c->h_tiles.data(), c->h_tiles.size() * sizeof(PdTile), cudaMemcpyHostToDevice, c->stream));
    c->h2d_bytes += c->h_tiles.size() * sizeof(PdTile);
    PD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
    PD_CUDA(c, cudaStreamSynchronize(c->stream));
    PD_CUDA(c, cudaEventElapsedTime(&c->ms_h2d, c->ev[0], c->ev[1]));
    c->uploaded = true; c->index_built = false;
    return 0;
}

extern "C" int pd_set_staging(pd_ctx * c, int pinned)
{
    if (!c) return PD_ERR_ARG;
    if (c->status) return c->status;
    c->pinned_staging = pinned != 0;
    return 0;
}

extern "C" int pd_set_unify(pd_ctx * c, const pd_unify_params * p)
{
    if (!c) return PD_ERR_ARG;
    if (c->status) return c->status;
    if (!p) { c->unify_on = false; return 0; }
    if (!(p->mean_stddev >= 0) || !(p->min_relative_window_cover >= 0)) return pd_fail(c, PD_ERR_ARG, "pd_set_unify: negative or NaN parameter");
    c->unify = *p; c->unify_on = true;
    return 0;
}

extern "C" int pd_contig_scan(pd_ctx * c, uint64_t first_window, uint64_t n_windows, pd_result * out)
{
    if (!c || !out) return PD_ERR_ARG;
    if (c->status) return c->status;
    if (c->device < 0) return pd_fail(c, PD_ERR_CUDA, "pd_contig_scan: host-only context (device = -1); the scan runs on a CUDA device only");
    float h2d = 0;
    if (!c->uploaded) { int rc = pd_contig_upload(c); if (rc) return rc; h2d = c->ms_h2d; }
    int rc = pd_run_scan(c, first_window, n_windows, out);
    if (rc == 0) { out->ms_h2d = h2d; out->ms_total += h2d; }
    return rc;
}

// ---------------------------------------------------------------------------------------------------------
// host-only validation hook: per-window sums from the PACKED image with the closed-form rule
// ---------------------------------------------------------------------------------------------------------
extern "C" int pd_debug_cap_replay(uint32_t window_buffer, uint32_t max_load, uint64_t n, const uint32_t * start,
                                   const uint32_t * end, uint8_t * stored)
{
    if (!window_buffer || (n && (!start || !end || !stored))) return PD_ERR_ARG;
    PdCapState cs;
    cs.start(window_buffer);
    for (uint64_t i = 0; i < n; ++i) {                              // the cap block of pd_contig_push
        const uint32_t b = start[i] / PD_WIN;
        const int64_t j = (int64_t)((uint64_t)b * PD_WIN / window_buffer);
        while (cs.seg < j) cs.next_segment(window_buffer);
        stored[i] = cs.admit(b, end[i] / PD_WIN, max_load);
    }
    return 0;
}

extern "C" int pd_debug_host_window_sums(pd_ctx * c, uint32_t rg, uint64_t first_window, uint64_t n_windows, int64_t * out)
{
    if (!c || !out || rg >= c->R) return PD_ERR_ARG;
    if (c->status) return c->status;
    if (!c->contig_open) return pd_fail(c, PD_ERR_ARG, "no open contig");
    if (c->dev_mode) return pd_fail(c, PD_ERR_ARG, "validation hook works on host-packed contigs only");
    int rc = pd_pack_contig(c);
    if (rc) return rc;
    memset(out, 0, sizeof(int64_t) * 3 * n_windows);
    const PdRgConst & k = c->rgc[rg];
    const PdHostRg & h = c->hrg[rg];
    const PdTile * off = &c->h_tiles[(size_t)rg * (c->NT + 1)];
    const uint64_t base = c->h_word_base[rg];
    auto add = [&](int64_t s, int64_t e, int32_t d, uint64_t pr) {
        for (int64_t w = std::max<int64_t>(s, (int64_t)first_window); w <= e && w < (int64_t)(first_window + n_windows); ++w) {
            int64_t * o = out + 3 * (w - first_window);
            o[0] += 1; o[1] += d; o[2] += (int64_t)(pr + c->grid.anchor);
        }
    };
    for (uint32_t t = 0; t < c->NT; ++t)
        for (uint64_t i = off[t].off - base; i < off[t + 1].off - base; ++i) {
            uint32_t w = h.words[i];
            if (pd_word_long(w)) continue;                         // pads and long read pairs
            uint64_t pr = (uint64_t)t * PD_TILE_BP + pd_word_pit(w);
            int64_t s, e;
            if (pd_interval(pr, pd_word_dev(w), k.inner_off, c->grid.window_buffer, s, e)) add(s, e, pd_word_dev(w), pr);
        }
    for (const PdLong & L : h.longs) add(L.s, L.e, L.dev, L.pos_rel);
    return 0;
}
