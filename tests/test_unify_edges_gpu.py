"""Device-side unifyCalls (pd_unify.cu) at the edges of its fixed capacities, through the pd_debug_unify probe: seeded
synthetic window calls go through the same kernels a scan's window calls go through, and the merged variants, their
per-sample rows and significant windows must equal the oracle's unify() on the same input (integers and rows exact, LR and
allele frequency within 1e-6). Ties are broken by window order on both sides (DESIGN 2), so they must match exactly.

The edges: PLAN_CAP (512 window calls per segment: the merge loop runs on shared-memory copies up to it, on global memory
past it or with PD_UNIFY_GLOBAL), EMIT_STAGE (1 024 in-range windows per variant: the median bisection re-reads the values
past it from global memory), the 32 lanes of the in-range ballot and of the PL / median loops, the emit grid (several
samples per warp once there are many variants) and the 1 024-thread scan of the per-segment variant counts."""
import numpy as np
import pytest

from popdel_b200 import api, simulate
from parity import assert_calls_equal

pytestmark = pytest.mark.gpu

SD = 40.0                                                   # mean insert-size stddev of the merge (2 sd / 4 sd rules)
SETTINGS = [(of, cover) for of in (False, True) for cover in (0.0, 0.5, 0.9)]     # (output_failed, min_relative_window_cover)
J = 20                                                      # position / length spread inside a cluster
FILTERS = [0] * 10 + [4, 4, 16, 1, 2, 8, 20, 32]            # bits 0-4 fail allPass, bit 5 does not


def _win(x):
    """First window position >= x."""
    return max(30, -(-int(x) // 30) * 30)


def _sort_key_order(pos, length, lr, idx):
    """Slots of lowerCall's order (position, length, LR descending), ties by window order: what both sides use."""
    return np.lexsort((idx, -lr, length, pos))


class _Gen:
    """Seeded window calls, built segment by segment in window order. A segment is a sequence of clusters that merge (nearby
    positions, similar lengths), chains that only checkAndExtend joins (span below the deletion length) and separators
    (short calls that merge with nothing)."""

    def __init__(self, seed, n_samples):
        self.rng = np.random.default_rng(seed)
        self.N = n_samples
        self.x = 1000                                       # next free position
        self.segs = []                                      # (tag, rows [wp, pos, len, end, lr, filter, cluster])
        self.exact = []                                     # clusters whose calls are all in range, for the median columns
        self.n_clusters = 0

    def segment(self, tag):
        self.segs.append((tag, []))

    def _add(self, wp, pos, length, end, cid=-1, filt=None, lr=None):
        r = self.rng
        self.segs[-1][1].append([int(wp), int(pos), int(length), int(end), float(r.uniform(3.0, 400.0)) if lr is None else lr,
                                 int(r.choice(FILTERS)) if filt is None else filt, cid])

    def separator(self):
        pos, length = self.x, int(self.rng.integers(40, 70))
        self._add(_win(pos + 30), pos, length, pos + length)
        self.x = pos + 300

    def cluster(self, k_in, k_out=0, exact=False):
        """k_in calls whose windows lie in the merged variant's range, k_out calls whose windows lie before it. With
        `exact` the k_in calls pass, so that the median position and length fall inside the cluster and the variant holds
        exactly k_in in-range windows when a separator or another cluster follows it."""
        r = self.rng
        P = _win(self.x + 200)
        m = int(r.integers(1, 4))                           # window calls per window (one per initial length)
        nwin = -(-k_in // m)
        L = max(int(r.integers(300, 3000)), 30 * nwin + 2 * J + 90)
        # in range: mp < P + J < wp and wp - 30 < P + L <= mp + ml
        wp = list(P + 60 + 30 * np.sort(r.integers(0, nwin, size=k_in)))
        w0 = _win(self.x)
        wp = list(np.sort(w0 + 30 * r.integers(0, (P - w0) // 30 + 1, size=k_out))) + wp      # wp <= P <= mp: out of range
        k = k_in + k_out
        pos = P + r.integers(0, J, size=k)
        length = L + r.integers(0, J, size=k)
        end = pos + length - r.integers(0, 4, size=k)
        lr = r.uniform(3.0, 400.0, size=k)
        filt = r.choice(FILTERS, size=k)
        cid = self.n_clusters
        self.n_clusters += 1
        first = _sort_key_order(pos, length, lr, np.arange(k))[0]
        if k >= 2:
            # exact tie on (position, length, LR) with the variant's first call, in another window: which of the two
            # represents the variant (window position, initial length, end) is decided by window order alone
            other = [j for j in range(k) if wp[j] != wp[first]]
            if other:
                j = int(r.choice(other))
                pos[j], length[j], lr[j] = pos[first], length[first], lr[first]
            if k >= 3 and r.random() < 0.5:                 # a tie on (position, length) alone: LR decides
                a, b = r.choice(k, size=2, replace=False)
                pos[b], length[b] = pos[a], length[a]
        if exact:
            filt[k_out:] = 0
        for j in range(k):
            self._add(wp[j], pos[j], length[j], end[j], cid, int(filt[j]), float(lr[j]))
        if exact:
            self.exact.append(cid)
        self.x = P + L + 2 * J + 200

    def chain(self, k):
        """Calls whose spans do not overlap (step > span) but lie within a deletion length of the variant's first call:
        checkAndExtend joins them and extends its end. Their windows are partly in range, possibly none."""
        r = self.rng
        P = _win(self.x + 200)
        L = int(r.integers(1500, 3000))
        span, step = L // 8, L // 6
        pos = P + step * np.arange(k) + r.integers(0, 5, size=k)
        last_end = int(pos[-1]) + span
        wp = np.sort(P + 30 * r.integers(0, (last_end - P) // 30 + 1, size=k))
        for j in range(k):
            self._add(wp[j], pos[j], L + int(r.integers(0, J)), int(pos[j]) + span)
        self.x = last_end + L + 400

    def random_segment(self, tag, n):
        """About n calls of clusters (mostly small, some past 32 in-range windows), chains and separators; cut to exactly
        n calls in window order, so the last cluster may be cut and end the segment."""
        r = self.rng
        self.segment(tag)
        calls = self.segs[-1][1]
        while len(calls) < n:
            u = r.random()
            if u < 0.55:
                k_in = int(r.integers(1, 9)) if r.random() < 0.85 else int(r.integers(30, 70))
                self.cluster(k_in, int(r.integers(0, 3)))
            elif u < 0.75:
                self.chain(int(r.integers(2, 12)))
            else:
                self.separator()
        self._close()
        del calls[n:]

    def exact_segment(self, tag, k_in):
        """One variant with exactly k_in in-range windows between two separators (k_in = 1: one more call out of range)."""
        self.segment(tag)
        self.separator()
        self.segs[-1][1][-1][5] = 0                          # the segment's first passing call (output_failed off)
        self.cluster(k_in, 1 if k_in == 1 else 0, exact=True)
        self.separator()
        self._close()

    def _close(self):
        """Window order; calls of one window in random order."""
        calls = self.segs[-1][1]
        o = np.lexsort((self.rng.random(len(calls)), [c[0] for c in calls]))
        calls[:] = [calls[i] for i in o]

    def build(self):
        """(calls, per_sample rows): PL below 2^16 with one zero per row (or all zero), LAD / DAD over the whole uint32
        range with duplicates; in the `exact` clusters LAD0 and LAD1 of every sample hold distinct values whose median is
        the variant's in-range window at index min(100, g - 1) and at index g - 1 (past EMIT_STAGE once g > 1 024)."""
        r = self.rng
        flat = [(tag, c) for tag, cs in self.segs for c in cs]
        n, N = len(flat), self.N
        calls = np.zeros(n, dtype=api.CALL_DTYPE)
        if n:
            a = np.array([c for _, c in flat], dtype=np.float64)
            calls["window_position"], calls["position"], calls["deletion_length"] = a[:, 0], a[:, 1], a[:, 2]
            calls["end_position"], calls["lr"], calls["filter"] = a[:, 3], a[:, 4], a[:, 5]
            calls["segment"] = [t for t, _ in flat]
            calls["initial_length"] = (a[:, 2] * r.uniform(0.5, 1.0, size=n)).astype(np.uint32)
            calls["iterations"] = r.integers(1, 16, size=n)
            calls["frequency"] = r.random(n)
        per = np.zeros((n, N, 13), dtype=np.uint32)
        scale = r.choice([100, 5000, 65535], size=(n, N, 1), p=[0.4, 0.4, 0.2])
        pl = (r.random((n, N, 3)) * scale).astype(np.uint32)
        pl[np.arange(n)[:, None], np.arange(N)[None, :], r.integers(0, 3, size=(n, N))] = 0
        pl[r.random((n, N)) < 0.05] = 0                     # low coverage: 0,0,0
        per[:, :, 0:3] = pl
        pool = np.concatenate([np.array([0, 0xFFFFFFFF], np.uint64), r.integers(0, 1 << 32, size=14, dtype=np.uint64)]).astype(np.uint32)
        fresh = r.integers(0, 1 << 32, size=(n, N, 10), dtype=np.uint64).astype(np.uint32)
        per[:, :, 3:13] = np.where(r.random((n, N, 10)) < 0.5, pool[r.integers(0, pool.size, size=(n, N, 10))], fresh)
        if n:
            cid = a[:, 6].astype(np.int64)
            for c in self.exact:
                idx = np.nonzero(cid == c)[0]
                wp, pos = calls["window_position"][idx], calls["position"][idx]
                idx = idx[wp > pos.max()]                   # the in-range windows
                inr = idx[_sort_key_order(calls["position"][idx], calls["deletion_length"][idx], calls["lr"][idx], idx)]
                g = inr.size
                for s in range(N):
                    for col, at in ((3, min(100, g - 1)), (4, g - 1)):
                        v = np.sort(r.choice(1 << 32, size=g, replace=False)).astype(np.uint32)
                        rest = np.delete(v, g // 2)
                        r.shuffle(rest)
                        per[inr, s, col] = np.insert(rest, at, v[g // 2])
        return calls, per


@pytest.fixture(scope="module")
def scanners():
    """One context per sample count (one read group per sample, copies of one processed histogram)."""
    samples, _ = simulate.simulate_cohort(seed=41, n_samples=1, contig_len=60_000, n_dels=0)
    params = api.CallParameters()
    rg = api.read_groups_from_headers(api.cohort_headers(samples), params)[0]
    made = {}

    def get(n_samples):
        if n_samples not in made:
            rgs = [api.ReadGroup(**{**rg.__dict__, "sample": s}) for s in range(n_samples)]
            made[n_samples] = api.Scanner(params, rgs, n_samples, device=0)
        return made[n_samples]

    yield get
    for sc in made.values():
        sc.close()


def _check(sc, calls, per, nseg, oracle_lib, settings=SETTINGS):
    """The probe against the oracle under every (output_failed, cover) setting; returns the variant counts."""
    counts = []
    for output_failed, cover in settings:
        what = f"output_failed={output_failed} cover={cover}"
        sc.set_unify(SD, cover, output_failed)
        got = sc.debug_unify(calls, per, nseg)
        ref_calls, ref_ps, ref_sig = oracle_lib.unify_segments(calls, per, SD, cover, output_failed)
        assert got["n_window_calls"] == len(calls), what
        try:
            assert_calls_equal(got["calls"], got["per_sample"], ref_calls, ref_ps)
        except AssertionError as e:
            raise AssertionError(f"{what}: {e}") from None
        assert np.array_equal(got["significant_windows"], ref_sig), what
        counts.append(len(ref_calls))
    return counts


@pytest.mark.parametrize("force_global", [False, True])
def test_segment_sizes(force_global, scanners, oracle_lib, monkeypatch):
    """Segments of 0, 1, 2, 31, 32, 33, 511, 512, 513 and 3 000 window calls in one input (the shared-memory merge up to
    PLAN_CAP = 512, global memory past it), plus segments in which every call fails, only the last call in lowerCall order
    passes, or only the one before it; with PD_UNIFY_GLOBAL every segment takes the global-memory path."""
    if force_global:
        monkeypatch.setenv("PD_UNIFY_GLOBAL", "1")
    g = _Gen(101, 3)
    sizes = [0, 1, 2, 31, 32, 33, 511, 512, 513, 3000]
    for tag, n in enumerate(sizes):
        if n:
            g.random_segment(tag, n)
    tag = len(sizes)
    for rule in ("none", "last", "second_last"):
        g.random_segment(tag, 40)
        cs = g.segs[-1][1]
        for c in cs:
            c[5] = 4
        if rule != "none":
            a = np.array(cs, dtype=np.float64)
            o = _sort_key_order(a[:, 1], a[:, 2], a[:, 4], np.arange(len(cs)))
            cs[o[-1 if rule == "last" else -2]][5] = 0
        tag += 1
    calls, per = g.build()
    counts = _check(scanners(3), calls, per, tag, oracle_lib)
    assert min(counts) > 100


def test_in_range_windows_per_variant(scanners, oracle_lib):
    """One variant with exactly 1, 31, 32, 33, 1 023, 1 024, 1 025 and 5 000 in-range windows per segment (the lanes of the
    in-range ballot and of the PL / median loops stride by 32; EMIT_STAGE = 1 024 values per warp are staged in shared
    memory). In two LAD columns the median is the window at index min(100, g - 1) and at index g - 1."""
    g = _Gen(102, 3)
    sizes = [1, 31, 32, 33, 1023, 1024, 1025, 5000]
    for tag, k in enumerate(sizes):
        g.exact_segment(tag, k)
    calls, per = g.build()
    sc = scanners(3)
    counts = _check(sc, calls, per, len(sizes), oracle_lib)
    assert counts == [len(sizes)] * len(SETTINGS)
    ref, _, _ = oracle_lib.unify_segments(calls, per, SD, 0.5, False)
    for t, v in enumerate(ref):                             # the in-range windows of each variant are the sizes asked for
        wp = calls["window_position"][calls["segment"] == t]
        assert int(((wp > v["position"]) & (wp - 30 < v["position"] + v["deletion_length"])).sum()) == sizes[t]


@pytest.mark.parametrize("n_samples", [1, 7, 9, 40, 257, 1100])
def test_sample_counts(n_samples, scanners, oracle_lib):
    """The emit grid is (variants, gy) with gy = min(ceil(N / 8), ceil(592 / variants)): with one or two variants every warp
    has one sample; with many variants gy < ceil(N / 8) and each warp loops over several samples, and the allele count adds
    up over the blocks of a variant before the last block writes the header."""
    sc = scanners(n_samples)
    few = _Gen(200 + n_samples, n_samples)
    few.segment(0)
    few.separator()
    few.cluster(40, 1, exact=True)
    few.separator()
    few.cluster(3, 0, exact=True)
    few.separator()
    few._close()
    calls, per = few.build()
    counts = _check(sc, calls, per, 1, oracle_lib)
    assert counts == [2] * len(SETTINGS)
    # many variants: enough that gy < ceil(N / 8) wherever N > 8; rows of n x N stay below ~40 MB
    many = _Gen(300 + n_samples, n_samples)
    n_var = 650 if n_samples <= 40 else (100 if n_samples <= 257 else 40)
    for tag in range(4):
        many.segment(tag)
        for _ in range(n_var // 4):
            many.cluster(int(many.rng.integers(2, 5)), 0, exact=True)
            many.separator()
        many._close()
    calls, per = many.build()
    counts = _check(sc, calls, per, 4, oracle_lib)
    total = min(counts)
    assert total >= n_var * 0.9
    if n_samples > 8:
        assert -(-592 // total) < -(-n_samples // 8)        # several samples per warp


@pytest.mark.parametrize("nseg", [1024, 1025, 1300, 2100])
def test_segment_counts(nseg, scanners, oracle_lib):
    """More segments than the 1 024 threads of k_unify_offsets: its scan carries the variant count of every earlier chunk.
    Calls in the first, the last and a few scattered segments; the others are empty."""
    g = _Gen(400 + nseg, 5)
    rng = np.random.default_rng(nseg)
    tags = sorted({0, nseg - 1, 1, 1023, *rng.integers(2, nseg - 1, size=6)} & set(range(nseg)))
    for t in tags:
        g.random_segment(t, int(rng.integers(20, 120)))
    calls, per = g.build()
    counts = _check(scanners(5), calls, per, nseg, oracle_lib)
    last = calls["segment"] >= 1024
    assert min(counts) > 0 and (nseg == 1024 or last.any())


def test_buffer_growth(oracle_lib, monkeypatch):
    """One context merges a small input, a large one (every device and mapped buffer grows) and a small one again."""
    monkeypatch.setenv("PD_UNIFY_CAP", "8")
    samples, _ = simulate.simulate_cohort(seed=41, n_samples=1, contig_len=60_000, n_dels=0)
    params = api.CallParameters()
    rg = api.read_groups_from_headers(api.cohort_headers(samples), params)[0]
    sc = api.Scanner(params, [api.ReadGroup(**{**rg.__dict__, "sample": s}) for s in range(4)], 4, device=0)
    try:
        inputs = []
        for seed, sizes in ((501, [12, 30]), (502, [600, 4000, 300]), (503, [25])):
            g = _Gen(seed, 4)
            for tag, n in enumerate(sizes):
                g.random_segment(tag, n)
            inputs.append((g.build(), len(sizes)))
        for (calls, per), nseg in inputs:
            _check(sc, calls, per, nseg, oracle_lib, settings=[(True, 0.5)])
    finally:
        sc.close()


def test_probe_refuses_what_it_cannot_merge():
    """PD_ERR_ARG without pd_set_unify, on a sample-sharded context and for segment tags out of order or >= nseg."""
    from test_host_logic import _cohort
    samples, params = _cohort("basic")
    rgs = api.read_groups_from_headers(api.cohort_headers(samples), params)
    calls = np.zeros(2, dtype=api.CALL_DTYPE)
    per = np.zeros((2, len(samples), 13), dtype=np.uint32)
    sc = api.Scanner(params, rgs, len(samples), device=0)
    try:
        with pytest.raises(api.ScanError, match=r"^\[-1\] pd_debug_unify: no unify settings"):
            sc.debug_unify(calls, per, 1)
    finally:
        sc.close()
    for tags, nseg in (([1, 0], 2), ([0, 2], 2)):
        sc = api.Scanner(params, rgs, len(samples), device=0)
        try:
            sc.set_unify(SD, 0.5, False)
            calls["segment"] = tags
            with pytest.raises(api.ScanError, match=r"^\[-1\] pd_debug_unify: segment tags"):
                sc.debug_unify(calls, per, nseg)
        finally:
            sc.close()
    grp = api.ShardGroup(samples, params, 2)
    try:
        sc = grp.scanners[0]
        sc.set_unify(SD, 0.5, False)
        calls["segment"] = 0
        with pytest.raises(api.ScanError, match=r"^\[-1\] pd_debug_unify: sample-sharded context"):
            sc.debug_unify(calls, per[:, :sc.n_samples], 1)
    finally:
        grp.close()
