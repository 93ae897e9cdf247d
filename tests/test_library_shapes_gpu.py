"""The device's read-pair walk (for_tile_batches, behind k_count, k_tile_q3, k_tile_cmask and k_tile_gather) against the
oracle's exact per-window active sets, for every cohort kind of test_host_logic._cohort and every push variant; and
window-range scans of the long-insert libraries, whose look-back spans up to 8 tiles, against the full scan."""
import numpy as np
import pytest

from popdel_b200 import api
from parity import assert_calls_equal, run_oracle
from test_host_logic import _cohort

pytestmark = pytest.mark.gpu

KINDS = ["basic", "mixedrg", "gap", "highcov", "longspan", "capborder", "capgap", "capspill", "capfar",
         "wideins", "matepair", "longins", "overlap", "megadel", "manyrg"]
PUSH_MODES = [False, True, "compact", "compact32", "device"]      # pd_contig_push, _pinned, _compact, _compact32, _device


@pytest.mark.parametrize("kind", KINDS)
def test_device_walk_reproduces_active_sets(kind, oracle_lib):
    """pd_debug_device_window_sums: count, sum of deviations and sum of positions of the read pairs the kernels' walk
    finds active in each window, per read group, equal the oracle's (= the reference's) active sets on every window.
    A walk that drops, repeats or misplaces a read pair fails here even when no call changes. On longins the range
    also starts inside a tile (window 5 000 of tile 156), below an 8-tile look-back."""
    samples, params = _cohort(kind)
    rgs = api.read_groups_from_headers(api.cohort_headers(samples), params)
    wins = None
    for mode in PUSH_MODES:
        sc = api.Scanner(params, rgs, len(samples), device=0)
        try:
            keep = api.push_cohort(sc, samples, mode)
            n = sc.window_count()
            if wins is None:
                _, _, n_ref, wins = run_oracle(samples, params, rgs, oracle_lib, window_sums=True, max_windows=n + 10)
                assert n_ref == n
            ranges = [(0, n)] + ([(5000, n - 5000)] if kind == "longins" else [])
            for first, count in ranges:
                for g in range(len(rgs)):
                    got = sc.debug_device_window_sums(g, first, count)
                    ref = wins[first:first + count, 1 + g, :]
                    bad = np.nonzero((got != ref).any(axis=1))[0]
                    assert bad.size == 0, (f"push {mode!r}, rg {g}, range from {first}: {bad.size} windows differ, first {first + bad[0]}: "
                                           f"{got[bad[0]]} vs {ref[bad[0]]}")
            del keep
        finally:
            sc.close()


@pytest.mark.parametrize("kind", ["longins", "matepair"])
def test_window_ranges_cut_through_long_lookback(kind, oracle_lib):
    """Scanning [0, 2 500), [2 500, 5 000) and [5 000, end) gives exactly the calls of the full scan, and those equal the
    oracle's. Both range starts lie inside a tile, with 6 (matepair) or 8 (longins) tiles of look-back before them."""
    samples, params = _cohort(kind)
    full, rgs = api.scan_cohort(samples, params)
    n = full["n_windows"]
    assert n > 6000
    parts = [api.scan_cohort(samples, params, first_window=a, n_windows=c)[0] for a, c in [(0, 2500), (2500, 2500), (5000, n - 5000)]]
    assert [p["n_windows"] for p in parts] == [2500, 2500, n - 5000]
    assert_calls_equal(np.concatenate([p["calls"] for p in parts]), np.concatenate([p["per_sample"] for p in parts]),
                       full["calls"], full["per_sample"], rtol=0)
    ref_calls, ref_ps, n_ref = run_oracle(samples, params, rgs, oracle_lib)
    assert n_ref == n
    assert_calls_equal(full["calls"], full["per_sample"], ref_calls, ref_ps)
    assert len(ref_calls) > 100
