"""Device-side unifyCalls on sample-sharded cohorts: after pd_set_unify on every rank, the collective scan returns the
merged variants (the same on every rank, allele frequency over the whole cohort) with the rows of the rank's own samples,
and they equal the oracle's unifyCalls applied to the window calls of the same sharded scan."""
import os
import time

import numpy as np
import pytest

from popdel_b200 import api, simulate
from parity import assert_calls_equal
from test_host_logic import _cohort

pytestmark = pytest.mark.gpu

# (highcov has two samples: a third rank would hold none; matepair, longins and megadel: segments past the merge loop's
# shared-memory slots and variants past the median's staged values)
KIND_WORLD = [(k, w) for k in ["basic", "mixedrg", "gap", "highcov", "longspan"] for w in (2, 3) if (k, w) != ("highcov", 3)] + \
    [("matepair", 2), ("longins", 2), ("megadel", 2)]


def _mean_stddev(rgs):
    return float(np.mean([r.stddev for r in rgs]))


def _oracle_merge(oracle_lib, raw, sd, cover, output_failed):
    return oracle_lib.unify_segments(raw["calls"], raw["per_sample"], sd, cover, output_failed)


@pytest.mark.parametrize("output_failed", [False, True])
@pytest.mark.parametrize("kind,world", KIND_WORLD)
def test_sharded_unify_equals_oracle_unify(kind, world, output_failed, oracle_lib):
    """Merged variants of the sharded scan == the oracle's unifyCalls on the window calls of the same sharded cohort."""
    samples, params = _cohort(kind)
    raw, rgs = api.scan_cohort_sample_sharded(samples, params, world)
    sd = _mean_stddev(rgs)
    uni, _ = api.scan_cohort_sample_sharded(samples, params, world,
                                            unify=dict(mean_stddev=sd, min_relative_window_cover=0.5, output_failed=output_failed))
    ref_calls, ref_ps, ref_sig = _oracle_merge(oracle_lib, raw, sd, 0.5, output_failed)
    assert uni["n_window_calls"] == len(raw["calls"]) and uni["n_windows"] == raw["n_windows"]
    assert_calls_equal(uni["calls"], uni["per_sample"], ref_calls, ref_ps)
    assert np.array_equal(uni["significant_windows"], ref_sig)
    assert 0 < len(uni["calls"]) < len(raw["calls"])


@pytest.mark.parametrize("kind,world", KIND_WORLD)
def test_sharded_unify_equals_single_context_unify(kind, world):
    """Sharded merge == single-context pd_set_unify on the same cohort (LR / AF within 1e-6: the sharded EM sums its
    statistics in rank order)."""
    samples, params = _cohort(kind)
    sd = _mean_stddev(api.read_groups_from_headers(api.cohort_headers(samples), params))
    for output_failed in (False, True):
        unify = dict(mean_stddev=sd, min_relative_window_cover=0.5, output_failed=output_failed)
        single, _ = api.scan_cohort(samples, params, unify=unify)
        uni, _ = api.scan_cohort_sample_sharded(samples, params, world, unify=unify)
        assert_calls_equal(uni["calls"], uni["per_sample"], single["calls"], single["per_sample"])
        assert np.array_equal(uni["significant_windows"], single["significant_windows"])
        assert uni["n_window_calls"] == single["n_window_calls"]


def test_sharded_unify_larger_cohort_buffer_growth_and_back(oracle_lib, monkeypatch):
    """40 samples over 4 ranks, EM chunks of 16 pairs and device-side call buffers that start at 8 calls (they grow between
    the EM chunks of the collective scan); cover 0.5 and 0.9 (the latter on the global-memory merge path). Every rank returns
    byte-equal variants and brings back fewer bytes than in window-call mode; switching back gives the window calls again."""
    samples, _ = simulate.simulate_cohort(seed=35, n_samples=40, contig_len=450_000, n_dels=6)
    params = api.CallParameters()
    monkeypatch.setenv("PD_UNIFY_CAP", "8")
    monkeypatch.setenv("PD_EM_CHUNK", "16")
    g = api.ShardGroup(samples, params, 4)
    try:
        raw = g.scan()
        sd = _mean_stddev(g.rgs)
        for cover in (0.5, 0.9):
            if cover == 0.9:
                monkeypatch.setenv("PD_UNIFY_GLOBAL", "1")
            g.set_unify(mean_stddev=sd, min_relative_window_cover=cover, output_failed=True)
            uni = g.scan()
            ref_calls, ref_ps, ref_sig = _oracle_merge(oracle_lib, raw, sd, cover, True)
            assert_calls_equal(uni["calls"], uni["per_sample"], ref_calls, ref_ps)
            assert np.array_equal(uni["significant_windows"], ref_sig)
            assert uni["n_window_calls"] == len(raw["calls"])
            p0 = uni["parts"][0]
            for r, p in enumerate(uni["parts"]):
                assert p["calls"].tobytes() == p0["calls"].tobytes() and p["significant_windows"].tobytes() == p0["significant_windows"].tobytes()
                assert p["d2h_bytes"] < raw["parts"][r]["d2h_bytes"], (r, p["d2h_bytes"], raw["parts"][r]["d2h_bytes"])
        assert len(ref_calls) >= 3
        g.set_unify(None)
        again = g.scan()
        assert_calls_equal(again["calls"], again["per_sample"], raw["calls"], raw["per_sample"], rtol=0)
    finally:
        g.close()


@pytest.mark.parametrize("case", ["rank0_only", "different_stddev"])
def test_sharded_unify_mismatched_settings_fail_on_every_rank(case):
    """Ranks whose unify settings differ would not enter the same exchanges: the scan fails on every rank with PD_ERR_ARG
    from its first collective, before any kernel runs, instead of waiting for the others."""
    samples, params = _cohort("basic")
    g = api.ShardGroup(samples, params, 2)
    try:
        g.scanners[0].set_unify(mean_stddev=50.0)
        if case == "different_stddev":
            g.scanners[1].set_unify(mean_stddev=51.0)
        t0 = time.perf_counter()
        with pytest.raises(api.ScanError) as e:
            g.scan()
        assert time.perf_counter() - t0 < 10.0
        assert str(e.value).startswith(f"[{-1}]")
        for sc in g.scanners:
            assert "unify settings differ between ranks" in sc.lib.pd_last_error(sc.ctx).decode()
    finally:
        g.close()


def _nccl_rank(rank, world, store, out_dir):
    import torch
    import torch.distributed as dist
    dist.init_process_group("gloo", init_method=f"file://{store}", rank=rank, world_size=world)
    try:
        samples, params = _cohort("mixedrg")
        sc, rgs, spr, mi = api.sample_shard_scanner(samples, params, world, rank, device=rank)
        uid = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(api.shard_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        sc.attach_nccl(rank, world, spr, mi, bytes(uid.numpy()))
        sc.set_unify(mean_stddev=_mean_stddev(rgs), min_relative_window_cover=0.5, output_failed=False)
        res = sc.scan()
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), calls=res["calls"], per_sample=res["per_sample"],
                 sig=res["significant_windows"], n_window_calls=res["n_window_calls"])
        sc.close()
    finally:
        dist.destroy_process_group()


def test_sharded_unify_nccl_transport(oracle_lib, tmp_path):
    """Two processes, one GPU each, attached with NCCL: the merged variants equal the oracle's merge of the window calls
    of the same cohort sharded over two in-process contexts."""
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    world = 2
    mp.spawn(_nccl_rank, args=(world, str(tmp_path / "store"), str(tmp_path)), nprocs=world, join=True)
    got = [np.load(tmp_path / f"rank{r}.npz") for r in range(world)]
    samples, params = _cohort("mixedrg")
    raw, rgs = api.scan_cohort_sample_sharded(samples, params, world)
    ref_calls, ref_ps, ref_sig = _oracle_merge(oracle_lib, raw, _mean_stddev(rgs), 0.5, False)
    for p in got[1:]:
        assert p["calls"].tobytes() == got[0]["calls"].tobytes() and np.array_equal(p["sig"], got[0]["sig"])
    assert int(got[0]["n_window_calls"]) == len(raw["calls"])
    per = np.concatenate([p["per_sample"] for p in got], axis=1)
    assert_calls_equal(got[0]["calls"], per, ref_calls, ref_ps)
    assert np.array_equal(got[0]["sig"], ref_sig)
    assert 0 < len(ref_calls) < len(raw["calls"])
