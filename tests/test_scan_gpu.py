"""GPU parity tests: the CUDA scan, called through the C ABI, against the CPU oracle on the same seeded cohorts.
Integer outputs (window positions, candidate and final lengths, iterations, PL/LAD/DAD/FL, filters, segments)
must be bit-exact; LR and allele frequency within 1e-6 relative (BASELINE.json north_star)."""
import numpy as np
import pytest

from popdel_b200 import api, simulate
from parity import assert_calls_equal, compare_scan_with_oracle, run_oracle
from test_host_logic import _cohort

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("kind", ["basic", "mixedrg", "gap", "highcov", "longspan", "capspill", "capfar",
                                  "wideins", "matepair", "longins", "overlap", "megadel", "manyrg"])
def test_scan_matches_oracle(kind, oracle_lib):
    samples, params = _cohort(kind)
    stats = compare_scan_with_oracle(samples, oracle_lib, params)
    assert stats["n_calls"] > 0
    assert stats["n_flagged"] < stats["n_windows"] // 4        # the screen prunes the bulk of the windows


def test_scan_window_wise_and_user_thresholds(oracle_lib):
    samples, _ = simulate.simulate_cohort(seed=31, n_samples=5, contig_len=240_000, n_dels=2)
    params = api.CallParameters(window_wise=True, min_init_len=150, min_len=120)
    stats = compare_scan_with_oracle(samples, oracle_lib, params)
    assert stats["n_calls"] > 0


def test_scan_somatic_and_iterations(oracle_lib):
    samples, _ = simulate.simulate_cohort(seed=32, n_samples=4, contig_len=210_000, n_dels=2)
    params = api.CallParameters(somatic=True, iterations=4)
    compare_scan_with_oracle(samples, oracle_lib, params)


def test_scan_no_deletions_and_empty_sample(oracle_lib):
    samples, _ = simulate.simulate_cohort(seed=33, n_samples=3, contig_len=120_000, n_dels=0)
    rg = samples[2].read_groups[0]
    rg.pos, rg.isize = rg.pos[:0], rg.isize[:0]                 # a sample without any read pair
    stats = compare_scan_with_oracle(samples, oracle_lib)
    assert stats["n_calls"] == 0


def test_scan_window_ranges_partition_the_contig(oracle_lib):
    """Window-range sharding (SURVEY.md 8e): scanning disjoint ranges yields exactly the calls of the full scan."""
    samples, _ = simulate.simulate_cohort(seed=34, n_samples=4, contig_len=450_000, n_dels=4)
    params = api.CallParameters()
    full, rgs = api.scan_cohort(samples, params)
    n = full["n_windows"]
    from popdel_b200.sharding import segment_aligned_ranges
    ranges = segment_aligned_ranges(n, params.window_buffer, 3)           # segment-aligned shards of 3 ranks
    assert [r[0] for r in ranges] == [0, 6667, 13334]
    parts = [api.scan_cohort(samples, params, first_window=a, n_windows=c)[0] for a, c in ranges]
    odd = [(0, 5000), (5000, 4000), (9000, n - 9000)]                     # arbitrary cuts work too
    parts2 = [api.scan_cohort(samples, params, first_window=a, n_windows=c)[0] for a, c in odd]
    assert_calls_equal(np.concatenate([p["calls"] for p in parts2]), np.concatenate([p["per_sample"] for p in parts2]),
                       full["calls"], full["per_sample"], rtol=0)
    calls = np.concatenate([p["calls"] for p in parts])
    ps = np.concatenate([p["per_sample"] for p in parts])
    assert sum(p["n_windows"] for p in parts) == n
    assert_calls_equal(calls, ps, full["calls"], full["per_sample"], rtol=0)
    ref_calls, ref_ps, _ = run_oracle(samples, params, rgs, oracle_lib)
    assert_calls_equal(full["calls"], full["per_sample"], ref_calls, ref_ps)


def test_larger_cohort(oracle_lib):
    """40 samples x 300 kbp: more samples than one warp, several candidates per window."""
    samples, _ = simulate.simulate_cohort(seed=35, n_samples=40, contig_len=300_000, n_dels=4)
    stats = compare_scan_with_oracle(samples, oracle_lib)
    assert stats["n_calls"] > 100


@pytest.mark.parametrize("kind", ["basic", "mixedrg", "gap", "highcov", "longspan", "capspill", "capfar",
                                  "wideins", "matepair", "longins", "overlap", "megadel", "manyrg"])
def test_device_packer_equals_host_packer(kind):
    """pd_contig_push_pinned / _compact / _device (device-side packing; host fallback when the coverage cap bites) == pd_contig_push."""
    samples, params = _cohort(kind)
    a, _ = api.scan_cohort(samples, params)
    # raw page-locked arrays / 5 and 4 bytes per read pair (pd_contig_push_compact, _compact32) / arrays already in device memory (pd_contig_push_device)
    for mode in (True, "compact", "compact32", "device"):
        b, _ = api.scan_cohort(samples, params, pinned=mode)
        assert a["n_windows"] == b["n_windows"] and a["n_flagged_windows"] == b["n_flagged_windows"]
        assert a["n_reads"] == b["n_reads"]
        assert_calls_equal(b["calls"], b["per_sample"], a["calls"], a["per_sample"], rtol=0)


def test_device_generator_equals_host_generator_and_device_push():
    """libpdsynth_cuda.so (SURVEY.md 8d: the on-device generator for cohorts that do not fit the host) writes the same read
    pairs as the host generator, and pd_contig_push_device packs them where they are: same calls as pd_contig_push."""
    import bench
    N, L, seed = 14, 420_000, 5
    ds, dl, gt = bench.plant(seed, N, L, 12.0)
    specs = bench.cohort_specs(seed, N, mixed=True)
    gen = api.SynthDevice(0)
    total, dp, dd, rg_start = gen.generate(seed, specs, 0, L, ds, dl, gt, N)
    pos_all, dev_all = gen.to_host(dp, total, np.uint32), gen.to_host(dd, total, np.int32)
    cohort, _ = bench.make_cohort(seed, N, L, 12.0, 4, mixed=True)
    assert int(rg_start[-1]) == total == sum(c[0].size for c in cohort)
    for g, c in enumerate(cohort):
        a, b = int(rg_start[g]), int(rg_start[g + 1])
        assert np.array_equal(pos_all[a:b], c[0]) and np.array_equal(dev_all[a:b], c[2]), f"read group {g}"
    # a window range of the same cohort: [first_pos, end_pos) is reproducible on its own
    t2, dp2, dd2, rs2 = gen.generate(seed, specs[:5], 120_000, 300_000, ds, dl, gt, N)
    p2 = gen.to_host(dp2, t2, np.uint32)
    for g in range(5):
        ref = cohort[g][0][(cohort[g][0] >= 120_000) & (cohort[g][0] < 300_000)]
        assert np.array_equal(p2[int(rs2[g]):int(rs2[g + 1])], ref)
    total, dp, dd, rg_start = gen.generate(seed, specs, 0, L, ds, dl, gt, N)
    params = api.CallParameters()
    rgs = api.read_groups_from_headers([[c[3] for c in cohort if c[4] == s] for s in range(N)], params)
    res = []
    for mode in ("host", "device"):
        sc = api.Scanner(params, rgs, N, device=0)
        sc.begin_contig(0)
        for g, c in enumerate(cohort):
            if mode == "host":
                sc.push(g, c[0], c[2])
            else:
                sc.push_device(g, int(rg_start[g + 1] - rg_start[g]), dp + 4 * int(rg_start[g]), dd + 4 * int(rg_start[g]))
        res.append(sc.scan())
        sc.close()
    gen.close()
    a, b = res
    assert a["n_windows"] == b["n_windows"] and a["n_reads"] == b["n_reads"] and len(a["calls"]) > 20
    assert_calls_equal(b["calls"], b["per_sample"], a["calls"], a["per_sample"], rtol=0)
    assert b["h2d_bytes"] < a["h2d_bytes"] // 100                     # nothing but the tables crossed PCIe


@pytest.mark.parametrize("n_samples,contig_len,env", [(150, 90_000, {}), (300, 70_000, {}), (150, 90_000, {"PD_EM_V2": "1"}),
                                                      (300, 70_000, {"PD_EM_V1": "1"}), (600, 50_000, {}), (1100, 45_000, {})])
def test_many_samples(n_samples, contig_len, env, oracle_lib, monkeypatch):
    """Larger cohorts: the fused pair-major kernel (<= 256 samples), the general pair-major kernels (PD_EM_V1) and the
    sample-major pipeline pd_em2.cu with one block per pair of 256 / 512 / 1024 threads and, beyond 1024 samples,
    several samples per thread."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    dels = [simulate.Deletion(30_000, 1200, np.random.default_rng(5).binomial(2, 0.3, size=n_samples))]
    samples, _ = simulate.simulate_cohort(seed=36, n_samples=n_samples, contig_len=contig_len, n_dels=0, dels=dels)
    stats = compare_scan_with_oracle(samples, oracle_lib)
    assert stats["n_calls"] > 20


@pytest.mark.parametrize("env", [{"PD_FORCE_SLOW": "7"}, {"PD_JOB_BATCH": "64", "PD_CJOB_ROWS": "7"}, {"PD_CJOB_ROWS": "1", "PD_EM_CHUNK": "5"},
                                 {"PD_EM_GENERAL": "1"}, {"PD_EM_V2": "1"}, {"PD_EM_V1": "1"}, {"PD_SCREEN2": "1"}, {"PD_SCREEN2": "0"},
                                 {"PD_SCREEN2": "1", "PD_FORCE_SLOW": "7", "PD_JOB_BATCH": "64"}])
@pytest.mark.parametrize("kind", ["basic", "mixedrg", "highcov", "matepair", "longins", "megadel"])
def test_scan_generic_paths_and_batching(kind, env, oracle_lib, monkeypatch):
    """The generic (no shared memory) Q3 / pool paths, small job batches, candidate-job sub-batches and EM chunks, and
    the general EM kernel give the same calls as the default configuration (all knobs are read per scan)."""
    samples, params = _cohort(kind)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    compare_scan_with_oracle(samples, oracle_lib, params)


@pytest.mark.parametrize("kind,world", [("basic", 2), ("mixedrg", 2), ("mixedrg", 3), ("highcov", 2), ("longspan", 3), ("matepair", 2)])
def test_sample_sharded_scan_equals_single_context(kind, world, oracle_lib):
    """Sample sharding (SURVEY.md 8e, config 5): `world` contexts of one process, each holding a block of the samples,
    exchange tile flags, Q3 values and the EM's per-iteration statistics (in-kernel, through peer memory). The merged
    result must equal the oracle and the single-context scan: integers bit-exact, LR / AF within 1e-6 relative (the
    cross-rank sums are taken in rank order, not in the single-context order)."""
    samples, params = _cohort(kind)
    merged, rgs = api.scan_cohort_sample_sharded(samples, params, world)
    single, _ = api.scan_cohort(samples, params)
    assert merged["n_windows"] == single["n_windows"] and merged["n_flagged_windows"] == single["n_flagged_windows"]
    assert_calls_equal(merged["calls"], merged["per_sample"], single["calls"], single["per_sample"])
    ref_calls, ref_ps, _ = run_oracle(samples, params, rgs, oracle_lib)
    assert_calls_equal(merged["calls"], merged["per_sample"], ref_calls, ref_ps)
    assert len(merged["calls"]) > 0


def test_sample_sharded_larger_cohort(oracle_lib):
    """40 samples over 4 contexts, several candidates per window, EM chunks of 16 pairs (several launches per scan)."""
    import os
    samples, _ = simulate.simulate_cohort(seed=35, n_samples=40, contig_len=300_000, n_dels=4)
    params = api.CallParameters()
    os.environ["PD_EM_CHUNK"] = "16"
    try:
        merged, rgs = api.scan_cohort_sample_sharded(samples, params, 4)
    finally:
        del os.environ["PD_EM_CHUNK"]
    ref_calls, ref_ps, _ = run_oracle(samples, params, rgs, oracle_lib)
    assert_calls_equal(merged["calls"], merged["per_sample"], ref_calls, ref_ps)
    assert len(merged["calls"]) > 100


def test_device_packer_with_empty_and_single_read_groups():
    """Pipelined device packer (8 copy groups) with fewer read groups than groups and with a read group without reads."""
    samples, _ = simulate.simulate_cohort(seed=33, n_samples=3, contig_len=120_000, n_dels=1)
    rg = samples[1].read_groups[0]
    rg.pos, rg.isize = rg.pos[:0], rg.isize[:0]
    params = api.CallParameters()
    a, _ = api.scan_cohort(samples, params)
    b, _ = api.scan_cohort(samples, params, pinned=True)
    assert a["n_windows"] == b["n_windows"] and a["n_reads"] == b["n_reads"]
    assert_calls_equal(b["calls"], b["per_sample"], a["calls"], a["per_sample"], rtol=0)
    one, _ = simulate.simulate_cohort(seed=37, n_samples=1, contig_len=90_000, n_dels=1)
    a, _ = api.scan_cohort(one, params)
    b, _ = api.scan_cohort(one, params, pinned=True)
    assert_calls_equal(b["calls"], b["per_sample"], a["calls"], a["per_sample"], rtol=0)


def _mean_stddev(rgs):
    return float(np.mean([r.as_dict()["stddev"] for r in rgs]))


@pytest.mark.parametrize("output_failed", [False, True])
@pytest.mark.parametrize("kind", ["basic", "mixedrg", "gap", "highcov", "longspan", "capspill", "capfar",
                                  "wideins", "matepair", "longins", "overlap", "megadel", "manyrg"])
def test_device_unify_equals_oracle_unify(kind, output_failed, oracle_lib):
    """pd_set_unify (unifyCalls on the device, SURVEY.md 8f rank 1): the merged variants equal the oracle's unifyCalls
    (utils_popdel.h:567-654, pinned against the reference's merged VCFs) applied to the same window calls. matepair,
    longins and megadel have segments of 973 to 8 446 window calls (past the merge loop's 512 shared-memory slots) and
    variants with more than 1 024 in-range windows (past the values a warp stages for the median)."""
    samples, params = _cohort(kind)
    raw, rgs = api.scan_cohort(samples, params)
    sd = _mean_stddev(rgs)
    uni, _ = api.scan_cohort(samples, params, unify=dict(mean_stddev=sd, min_relative_window_cover=0.5, output_failed=output_failed))
    ref_calls, ref_ps, ref_sig = oracle_lib.unify_segments(raw["calls"], raw["per_sample"], sd, 0.5, output_failed)
    assert uni["n_window_calls"] == len(raw["calls"]) and uni["n_windows"] == raw["n_windows"]
    assert_calls_equal(uni["calls"], uni["per_sample"], ref_calls, ref_ps)
    assert np.array_equal(uni["significant_windows"], ref_sig)
    assert 0 < len(ref_calls) < len(raw["calls"])


def test_device_unify_larger_cohort_and_buffer_growth(oracle_lib, monkeypatch):
    """40 samples, several segments, tight window cover; the device-side call buffers start tiny and grow per EM chunk."""
    samples, _ = simulate.simulate_cohort(seed=35, n_samples=40, contig_len=450_000, n_dels=6)
    params = api.CallParameters()
    raw, rgs = api.scan_cohort(samples, params)
    sd = _mean_stddev(rgs)
    monkeypatch.setenv("PD_UNIFY_CAP", "8")
    monkeypatch.setenv("PD_EM_CHUNK", "16")
    for cover in (0.5, 0.9):
        if cover == 0.9:
            monkeypatch.setenv("PD_UNIFY_GLOBAL", "1")     # the path for segments with more window calls than the shared-memory copies hold
        uni, _ = api.scan_cohort(samples, params, unify=dict(mean_stddev=sd, min_relative_window_cover=cover, output_failed=True))
        ref_calls, ref_ps, ref_sig = oracle_lib.unify_segments(raw["calls"], raw["per_sample"], sd, cover, True)
        assert_calls_equal(uni["calls"], uni["per_sample"], ref_calls, ref_ps)
        assert np.array_equal(uni["significant_windows"], ref_sig)
    assert len(ref_calls) >= 3
    # back to window calls on the same context kind
    again, _ = api.scan_cohort(samples, params)
    assert_calls_equal(again["calls"], again["per_sample"], raw["calls"], raw["per_sample"], rtol=0)
