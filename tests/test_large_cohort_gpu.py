"""Cohorts past the shared-memory budget of the candidate step (51 700 samples) and past 65 535 samples per launch grid
row: the instance of k_candidates that reads the Q3s from global memory (pd_debug_candidates against a restatement of
initialize_deletion_lengths, and whole scans through it with PD_CAND_GLOBAL=1), and one 70 000-sample cohort end to end."""
import time

import numpy as np
import pytest

from popdel_b200 import api, simulate
from parity import assert_calls_equal, compare_scan_with_oracle, run_oracle
from test_host_logic import _cohort

pytestmark = pytest.mark.gpu

SMEM_SAMPLES = 51_700          # the largest cohort whose Q3s the shared-memory instance holds (npad * 4 <= 202 KB)


def restated_candidates(q3, state, min_init):
    """initialize_deletion_lengths (SURVEY App. F, genotype_deletion_popdel_call.h:58-86): sort the Q3s of the samples that
    have one, chain neighbours closer than 50, keep a chain's int mean (C's truncating division of an int sum) when it
    exceeds the smallest threshold among the chain's RANKS in the sorted array."""
    v = np.sort(q3[state == 2]).astype(np.int64)
    if v.size == 0:
        return np.zeros(0, np.int32)
    starts = np.r_[0, np.nonzero(np.diff(v) >= 50)[0] + 1]
    sums = np.add.reduceat(v, starts)
    sums = (sums + 2**31) % 2**32 - 2**31                            # int accumulator
    cnts = np.diff(np.r_[starts, v.size])
    means = np.sign(sums) * (np.abs(sums) // cnts)                    # truncation toward zero
    thr = np.minimum.reduceat(np.asarray(min_init, np.int64)[:v.size], starts)
    return means[means > thr].astype(np.int32)


def _windows(n, rng):
    """Q3 / state rows of the probe's window kinds for a cohort of n samples: [n_windows, n] each."""
    rows = []

    def add(vals, p_has=0.8, garbage=True):
        st = np.where(rng.random(n) < p_has, 2, rng.integers(0, 2, n)).astype(np.uint8)
        q = np.asarray(vals, np.int64)
        if garbage:                                                   # a Q3 without state 2 must not count
            q = np.where(st == 2, q, rng.integers(-10**6, 10**6, n))
        rows.append((q.astype(np.int32), st))

    add(400 + rng.integers(0, 40, n))                                                 # one cluster
    add(rng.integers(-400, 900, n))                                                   # negative values, a dense range
    add(rng.choice(np.array([-250, -201, -152, 100, 149, 199, 300, 350, 399]), n))   # ties; chains 49 and 50 apart
    add(np.where(rng.random(n) < 0.001, rng.choice([-70_000, 70_000], n), rng.integers(200, 260, n)))   # range beyond 65 536
    add(np.where(np.arange(n) % 97 == 0, rng.integers(300_000, 300_100, n), rng.integers(-30, 30, n)))  # range, far chain
    i = np.arange(n)
    add(50 * (i % 1_100) - 30_000)                                                    # > 1 024 clusters 50 apart, inside the bitmap range
    add(49 * (i % 1_100) - 20_000)                                                    # one chain of steps of 49
    add(100 * (i % 1_100) + 49 * ((i // 1_100) % 2))                                 # > 1 024 pairs 49 apart, range beyond 65 536
    add(rng.integers(0, 500, n), p_has=0.0)                                           # no sample has a Q3
    add(rng.integers(100, 5_000, n), p_has=0.3)                                       # mixed state bytes, sparse
    q = np.stack([r[0] for r in rows])
    s = np.stack([r[1] for r in rows])
    return q, s


@pytest.fixture(scope="module")
def read_group_template():
    samples, _ = simulate.simulate_cohort(seed=61, n_samples=1, contig_len=40_000, n_dels=0)
    params = api.CallParameters()
    return params, api.read_groups_from_headers(api.cohort_headers(samples), params)[0]


def _probe_scanner(n, template, seed):
    """A context of n single-read-group samples with thresholds that differ by rank (read group)."""
    params, rg = template
    mi = np.random.default_rng([seed, 1]).integers(40, 400, n)
    rgs = [api.ReadGroup(**{**rg.__dict__, "sample": s, "min_init_del_len": int(mi[s])}) for s in range(n)]
    return api.Scanner(params, rgs, n, device=0), mi


@pytest.mark.parametrize("n", [1, 2, 31, SMEM_SAMPLES, SMEM_SAMPLES + 1, 65_536, 200_000])
def test_probe_equals_restatement(n, read_group_template, monkeypatch):
    """pd_debug_candidates == the restatement on every window kind; at sizes the shared-memory instance can hold, the
    global-memory instance (PD_CAND_GLOBAL=1) gives the same candidates as the shared-memory one."""
    rng = np.random.default_rng([71, n])
    q3, st = _windows(n, rng)
    sc, mi = _probe_scanner(n, read_group_template, n)
    try:
        want = [restated_candidates(q3[w], st[w], mi) for w in range(q3.shape[0])]
        assert sum(c.size for c in want) > 0
        modes = ["0", "1"] if n <= SMEM_SAMPLES else ["0"]            # above the budget the global instance runs either way
        for mode in modes:
            monkeypatch.setenv("PD_CAND_GLOBAL", mode)
            got = sc.debug_candidates(q3, st)
            for w in range(q3.shape[0]):
                assert np.array_equal(got[w], want[w]), f"PD_CAND_GLOBAL={mode}, window {w}: {got[w][:8]} vs {want[w][:8]}"
    finally:
        sc.close()


def test_probe_refuses_host_only_and_sharded(read_group_template):
    params, rg = read_group_template
    q3 = np.zeros((1, 2), np.int32)
    st = np.full((1, 2), 2, np.uint8)
    rgs = [api.ReadGroup(**{**rg.__dict__, "sample": s}) for s in range(2)]
    host = api.Scanner(params, rgs, 2, device=-1)
    try:
        with pytest.raises(api.ScanError, match=r"\[-1\].*host-only"):
            host.debug_candidates(q3, st)
    finally:
        host.close()
    samples, params = _cohort("basic")
    g = api.ShardGroup(samples, params, 2)
    try:
        n = g.scanners[0].n_samples
        with pytest.raises(api.ScanError, match=r"\[-1\].*sample-sharded"):
            g.scanners[0].debug_candidates(np.zeros((1, n), np.int32), np.full((1, n), 2, np.uint8))
    finally:
        g.close()


@pytest.mark.parametrize("kind", ["basic", "mixedrg", "highcov", "megadel", "longins"])
def test_global_instance_scan_equals_oracle(kind, oracle_lib, monkeypatch):
    """Whole scans with the global-memory instance of k_candidates (megadel: its sorting fallback) equal the oracle."""
    monkeypatch.setenv("PD_CAND_GLOBAL", "1")
    samples, params = _cohort(kind)
    stats = compare_scan_with_oracle(samples, oracle_lib, params)
    assert stats["n_calls"] > 0


def test_global_instance_sharded_matepair_equals_oracle(oracle_lib, monkeypatch):
    monkeypatch.setenv("PD_CAND_GLOBAL", "1")
    samples, params = _cohort("matepair")
    res, rgs = api.scan_cohort_sample_sharded(samples, params, 2)
    ref_calls, ref_ps, n_windows = run_oracle(samples, params, rgs, oracle_lib)
    assert res["n_windows"] == n_windows and len(ref_calls) > 0
    assert_calls_equal(res["calls"], res["per_sample"], ref_calls, ref_ps)


# ---- one cohort past both limits: 70 000 samples (> 51 700 for the candidate step, > 65 535 grid rows of k_count and of
# the sample-major EM's read-group grid) over a short contig with one planted deletion
N_LARGE = 70_000
CONTIG = 13_000


def assert_large_calls_equal(got, ref, pl_step=1):
    """The parity rules of tests/parity.py, except that a PL may differ by one in a few rows: a PL is a rounded log10 of
    double likelihoods whose last bits depend on the order of the sums over the samples, and over millions of rows a few
    of them sit on a rounding border (the fused and the sample-major EM of this library already differ there at 20 000
    samples). Every other per-sample value is exact. (Merged variants sum the PLs of their windows and subtract the
    smallest: pl_step=2.)"""
    assert_calls_equal(got["calls"], np.zeros(0), ref["calls"], np.zeros(0))
    a, b = got["per_sample"].astype(np.int64), ref["per_sample"].astype(np.int64)
    assert a.shape == b.shape
    assert np.array_equal(a[:, :, 3:], b[:, :, 3:]), "per-sample LAD/DAD/FL differ"
    d = np.abs(a[:, :, :3] - b[:, :, :3])
    assert d.max(initial=0) <= pl_step, "a PL differs by more than the rounding of its likelihoods allows"
    rows = np.count_nonzero(d.any(axis=2))
    assert rows <= max(1, a.shape[0] * a.shape[1] // 100_000), f"{rows} of {a.shape[0] * a.shape[1]} rows have a PL off"


@pytest.fixture(scope="module")
def large_cohort():
    t0 = time.time()
    rng = np.random.default_rng(81)
    gt = rng.choice(np.array([0, 1, 2], np.uint8), N_LARGE, p=[0.7, 0.2, 0.1])
    specs = [[simulate.ReadGroupSpec(name=f"rg{s}", coverage=8)] for s in range(N_LARGE)]
    samples, _ = simulate.simulate_cohort(seed=82, n_samples=N_LARGE, contig_len=CONTIG, n_dels=0,
                                          dels=[simulate.Deletion(6_000, 1_200, gt)], rg_specs=specs)
    print(f"large cohort: {N_LARGE} samples generated in {time.time() - t0:.1f} s")
    return samples, api.CallParameters()


@pytest.fixture(scope="module")
def large_single(large_cohort):
    samples, params = large_cohort
    return api.scan_cohort(samples, params)


def test_large_cohort_single_context_equals_oracle(large_cohort, large_single, oracle_lib):
    samples, params = large_cohort
    res, rgs = large_single
    ref_calls, ref_ps, n_windows = run_oracle(samples, params, rgs, oracle_lib, max_calls=400)
    assert res["n_windows"] == n_windows
    assert len(ref_calls) > 0 and len(res["calls"]) > 0
    assert_large_calls_equal(res, dict(calls=ref_calls, per_sample=ref_ps))


def test_large_cohort_sharded_equals_single_context(large_cohort, large_single):
    samples, params = large_cohort
    single, rgs = large_single
    sharded, _ = api.scan_cohort_sample_sharded(samples, params, 2)
    assert sharded["n_windows"] == single["n_windows"] and len(single["calls"]) > 0
    assert_large_calls_equal(sharded, single)
    unify = dict(mean_stddev=float(np.mean([r.stddev for r in rgs])), min_relative_window_cover=0.5, output_failed=False)
    u_single, _ = api.scan_cohort(samples, params, unify=unify)
    u_sharded, _ = api.scan_cohort_sample_sharded(samples, params, 2, unify=unify)
    assert len(u_single["calls"]) > 0
    assert_large_calls_equal(u_sharded, u_single, pl_step=2)
    assert np.array_equal(u_sharded["significant_windows"], u_single["significant_windows"])
