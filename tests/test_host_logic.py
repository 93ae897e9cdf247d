"""CPU-only tests of the product's host logic: the C ABI loads and exports what include/popdel_b200.h declares,
histogram preprocessing equals the oracle, and the packed tile layout + closed-form activity rule reproduce the
oracle's (= the reference's) per-window active sets. No scan is run here: the scan has no CPU path."""
import os
import re

import numpy as np
import pytest

from popdel_b200 import api, simulate

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    lib = api.load_library()
    header = open(os.path.join(ROOT, "include", "popdel_b200.h")).read()
    declared = set(re.findall(r"\b(pd_[a-z_0-9]+)\s*\(", header)) - {"pd_ctx"}
    assert declared == set(api.EXPORTS)
    for name in declared:
        assert getattr(lib, name) is not None


def test_generator_libraries_export_every_declared_symbol():
    """include/pdsynth.h: the host generator (libpdsynth.so) and its device-side twin (libpdsynth_cuda.so, loads without a GPU)."""
    import ctypes as C
    header = open(os.path.join(ROOT, "include", "pdsynth.h")).read()
    declared = set(re.findall(r"\b(pd_synth_[a-z_]+|pdsynth_dev_[a-z_]+)\s*\(", header))
    assert declared == {"pd_synth_read_group", "pdsynth_dev_create", "pdsynth_dev_destroy", "pdsynth_dev_generate", "pdsynth_dev_copy_to_host"}
    host = C.CDLL(os.path.join(ROOT, "popdel_b200", "libpdsynth.so"))
    dev = C.CDLL(os.path.join(ROOT, "popdel_b200", "libpdsynth_cuda.so"))
    for name in declared:
        assert getattr(host if name.startswith("pd_synth_") else dev, name) is not None


def test_compact_encode_round_trip():
    """pd_contig_push_compact's input form: 16-bit position remainders per 65 536-bp block + 24-bit deviations."""
    rng = np.random.default_rng(11)
    pos = np.sort(rng.integers(990, 400_000, size=5000)).astype(np.uint32)
    pos[:3] = 990
    dev = rng.integers(-400, 19_000, size=5000).astype(np.int32)
    lo, d24, blk = api.compact_encode(pos, dev)
    assert lo.size == 5000 and d24.size == 15000 and blk[0] == 0 and blk[-1] == 5000
    back = np.zeros(5000, np.uint32)
    for b in range(blk.size - 1):
        back[blk[b]:blk[b + 1]] = (b << 16) | lo[blk[b]:blk[b + 1]].astype(np.uint32)
    assert np.array_equal(back, pos)
    u = d24.reshape(-1, 3).astype(np.uint32)
    d = (u[:, 0] | (u[:, 1] << 8) | (u[:, 2] << 16)).astype(np.int64)
    d = np.where(d >= 1 << 23, d - (1 << 24), d)
    assert np.array_equal(d, dev)
    # 4-byte form (pd_contig_push_compact32): 8-bit position remainders per 256-bp block, 24-bit deviations in one word
    w, blk8 = api.compact32_encode(pos, dev)
    assert w.size == 5000 and blk8[0] == 0 and blk8[-1] == 5000 and blk8.size == (int(pos[-1]) >> 8) + 2
    back = np.zeros(5000, np.uint32)
    for b in range(blk8.size - 1):
        back[blk8[b]:blk8[b + 1]] = (b << 8) | (w[blk8[b]:blk8[b + 1]] & 0xFF)
    assert np.array_equal(back, pos) and np.array_equal(w.view(np.int32) >> 8, dev)


def test_process_histogram_equals_oracle(oracle_lib):
    rng = np.random.default_rng(3)
    for mu, sd, rl in [(500, 50, 150), (350, 30, 100), (550, 80, 150), (300, 100, 125)]:
        isz = np.rint(rng.normal(mu, sd, size=200000)).astype(np.int64)
        med = int(np.median(isz))
        lo, hi = max(1, int(np.floor(med - 3 * sd))), int(np.ceil(med + 3 * sd)) + 1
        counts = np.bincount(isz[(isz >= lo) & (isz < hi)] - lo, minlength=hi - lo).astype(np.float64)
        for smoothing in (True, False):
            a = api.process_histogram(counts, lo, med, rl, smoothing, 500)
            b = oracle_lib.process_histogram(counts, lo, med, rl, smoothing, 500)
            assert np.array_equal(a[0], b[0]) and a[1:] == b[1:]


def _cohort(kind):
    if kind == "basic":
        return simulate.simulate_cohort(seed=21, n_samples=3, contig_len=430_000, n_dels=2)[0], api.CallParameters()
    if kind == "mixedrg":
        specs = simulate.mixed_rg_specs(4, 4)
        return simulate.simulate_cohort(seed=22, n_samples=4, contig_len=260_000, n_dels=2, rg_specs=specs)[0], api.CallParameters()
    if kind == "gap":
        dels = [simulate.Deletion(100_000, 1800, np.array([1, 2, 1])), simulate.Deletion(700_000, 900, np.array([2, 0, 1]))]
        samples, _ = simulate.simulate_cohort(seed=23, n_samples=3, contig_len=800_000, n_dels=0, dels=dels)
        for k, s in enumerate(samples):
            for rg in s.read_groups:
                keep = ~((rg.pos >= 150_000) & (rg.pos < 610_000))
                if k == 0:
                    keep &= ~((rg.pos >= 20_000) & (rg.pos < 60_000))
                rg.pos, rg.isize = rg.pos[keep], rg.isize[keep]
        return samples, api.CallParameters()
    if kind == "highcov":
        samples, _ = simulate.simulate_cohort(seed=24, n_samples=2, contig_len=230_000, n_dels=1)
        spec = simulate.ReadGroupSpec(name="burst", coverage=400.0)
        extra, _ = simulate.simulate_cohort(seed=25, n_samples=1, contig_len=230_000, n_dels=0, rg_specs=[[spec]])
        e = extra[0].read_groups[0]
        m = (e.pos >= 90_000) & (e.pos < 120_000)
        rg = samples[0].read_groups[0]
        p, i = np.concatenate([rg.pos, e.pos[m]]), np.concatenate([rg.isize, e.isize[m]])
        o = np.lexsort((i, p))
        rg.pos, rg.isize = p[o], i[o]
        return samples, api.CallParameters()
    if kind in ("capborder", "capgap", "capspill"):
        # the active-coverage cap across segment borders (borders at anchor + k * 200 000):
        #  capborder: a 400x burst that runs over a border, so the first add() of the new segment happens with the cap active
        #  capgap:    the read group then sits out one / two whole segments (correctConsecutiveSwitch zeroes the counter)
        #  capspill:  the burst carries a large deletion right before the border (many spill-over end entries)
        dels = [simulate.Deletion(198_500, 1200, np.array([2, 1]))] if kind == "capspill" else []
        samples, _ = simulate.simulate_cohort(seed=27, n_samples=2, contig_len=1_030_000, n_dels=0, dels=dels)
        spec = simulate.ReadGroupSpec(name="burst", coverage=400.0)
        extra, _ = simulate.simulate_cohort(seed=28, n_samples=1, contig_len=1_030_000, n_dels=0, dels=dels[:1] and
                                            [simulate.Deletion(198_500, 1200, np.array([2]))], rg_specs=[[spec]])
        e = extra[0].read_groups[0]
        m = ((e.pos >= 185_000) & (e.pos < 215_000)) | ((e.pos >= 399_000) & (e.pos < 401_500)) | ((e.pos >= 795_000) & (e.pos < 830_000))
        rg = samples[0].read_groups[0]
        keep = np.ones(rg.pos.size, bool)
        if kind == "capgap":
            keep &= ~((rg.pos >= 215_000) & (rg.pos < 399_000))            # only bursts in segments 1 and 2, nothing in segment 3
            keep &= ~((rg.pos >= 401_500) & (rg.pos < 795_000))
            m &= ~((e.pos >= 200_000) & (e.pos < 215_000)) | (e.pos >= 399_000)
        p, i = np.concatenate([rg.pos[keep], e.pos[m]]), np.concatenate([rg.isize[keep], e.isize[m]])
        o = np.lexsort((i, p))
        rg.pos, rg.isize = p[o], i[o]
        return samples, api.CallParameters()
    if kind == "capfar":
        # read pairs spanning more than a segment keep the cursor of getEndCount inside their end set, so the reference's
        # activeLoad counter stops seeing the read pairs that close in the following sets and sticks at maxLoad
        samples, _ = simulate.simulate_cohort(seed=29, n_samples=2, contig_len=700_000, n_dels=2)
        spec = simulate.ReadGroupSpec(name="burst", coverage=400.0)
        extra, _ = simulate.simulate_cohort(seed=30, n_samples=1, contig_len=700_000, n_dels=0, rg_specs=[[spec]])
        e = extra[0].read_groups[0]
        m = ((e.pos >= 350_000) & (e.pos < 365_000)) | ((e.pos >= 520_000) & (e.pos < 530_000))
        rg = samples[0].read_groups[0]
        far_pos = np.array([150_003, 150_950, 188_000], dtype=rg.pos.dtype)
        far_isz = np.array([262_000, 255_000, 420_000], dtype=rg.isize.dtype)
        p, i = np.concatenate([rg.pos, e.pos[m], far_pos]), np.concatenate([rg.isize, e.isize[m], far_isz])
        o = np.lexsort((i, p))
        rg.pos, rg.isize = p[o], i[o]
        return samples, api.CallParameters()
    if kind == "longspan":
        # a large deletion (long read pairs in the wide list) crossing a segment border
        dels = [simulate.Deletion(196_000, 9000, np.array([1, 2, 1]))]
        return simulate.simulate_cohort(seed=26, n_samples=3, contig_len=260_000, n_dels=0, dels=dels)[0], api.CallParameters()
    if kind in _LIBRARY_KINDS:
        return _library_cohort(kind), api.CallParameters()
    raise KeyError(kind)


# Libraries other than ~500 +- 80 bp / 150-bp reads. The insert-size distribution decides the look-back of the packed
# stream (pd_create: ceil(((29 + median - 2 readLen + 8 sd) / 30 + 2) / 32) tiles, at most PD_MAX_LOOKBACK_TILES = 8),
# how many read pairs go to the wide list and how many rows the likelihood tables have (hist_end - hist_start):
#   wideins   900 +- 150, 100-bp reads: look-back 3
#   matepair  2 500 +- 400: look-back 6, a 20-kbp hole in one sample (tiles without read pairs inside the look-back),
#             2 401-row tables (the sample-major EM with more than 48 KB of dynamic shared memory)
#   longins   8 000 +- 1 200: look-back clamped at 8, most read pairs in the wide list, 7 201-row tables (sample-major EM off)
#   overlap   330 +- 60 at 50x with a quarter of the insert sizes in [0, 300): overlapping reads, inner distance clamped to 0,
#             deviations down to -median
#   megadel   a 1.1-Mbp deletion: deviations above PD_DEV_MAX (clamped in the stream word, kept in the wide list) and Q3
#             values beyond the presence bitmap of the candidate step
#   manyrg    10 read groups per sample with mixed read lengths: more read groups than the gather's fast path holds
_LIBRARY_KINDS = ("wideins", "matepair", "longins", "overlap", "megadel", "manyrg")


def _library_cohort(kind):
    spec = simulate.ReadGroupSpec

    def genotypes(n, p):
        return np.random.default_rng(5).binomial(2, p, size=n)

    if kind == "wideins":
        specs = [[spec(name=f"rg{s}", mu=900, sigma=150, read_length=100, coverage=20)] for s in range(6)]
        dels = [simulate.Deletion(100_000, 2500, genotypes(6, 0.5))]
        return simulate.simulate_cohort(seed=51, n_samples=6, contig_len=200_000, n_dels=0, dels=dels, rg_specs=specs)[0]
    if kind == "matepair":
        specs = [[spec(name=f"rg{s}", mu=2500, sigma=400, coverage=8)] for s in range(6)]
        dels = [simulate.Deletion(100_000, 5000, genotypes(6, 0.5))]
        samples = simulate.simulate_cohort(seed=51, n_samples=6, contig_len=200_000, n_dels=0, dels=dels, rg_specs=specs)[0]
        rg = samples[2].read_groups[0]
        keep = ~((rg.pos >= 40_000) & (rg.pos < 60_000))
        rg.pos, rg.isize = rg.pos[keep], rg.isize[keep]
        return samples
    if kind == "longins":
        specs = [[spec(name=f"rg{s}", mu=8000, sigma=1200, coverage=3)] for s in range(6)]
        dels = [simulate.Deletion(130_000, 9000, genotypes(6, 0.5))]
        return simulate.simulate_cohort(seed=51, n_samples=6, contig_len=260_000, n_dels=0, dels=dels, rg_specs=specs)[0]
    if kind == "overlap":
        # 50x: at 30x a hom carrier keeps a single active read pair right after the deletion, and its reference shift is
        # the x87 artefact of DESIGN 2 (the shift quotient lands on the deviation or one ulp below it)
        specs = [[spec(name=f"rg{s}", mu=330, sigma=60, coverage=50)] for s in range(4)]
        dels = [simulate.Deletion(60_000, 800, genotypes(4, 0.5))]
        samples = simulate.simulate_cohort(seed=51, n_samples=4, contig_len=120_000, n_dels=0, dels=dels, rg_specs=specs)[0]
        rng = np.random.default_rng(52)
        for s in samples:
            rg = s.read_groups[0]
            short = rng.random(rg.pos.size) < 0.25              # the simulator clips insert sizes at 2 * readLen
            isz = np.where(short, rng.integers(0, 300, size=rg.pos.size), rg.isize).astype(np.int32)
            o = np.lexsort((isz, rg.pos))
            rg.pos, rg.isize = rg.pos[o], isz[o]
            simulate.finalize_histogram(rg)
        return samples
    if kind == "megadel":
        dels = [simulate.Deletion(200_000, 1_100_000, genotypes(4, 0.5))]
        return simulate.simulate_cohort(seed=51, n_samples=4, contig_len=1_500_000, n_dels=0, dels=dels)[0]
    if kind == "manyrg":
        specs = [[spec(name=f"s{s}_rg{j}", mu=(350, 450, 550)[j % 3], sigma=(30, 50, 80)[(j + s) % 3],
                       read_length=(100, 125, 150)[(j // 3 + s) % 3], coverage=15) for j in range(10)] for s in range(3)]
        return simulate.simulate_cohort(seed=51, n_samples=3, contig_len=150_000, n_dels=2, rg_specs=specs)[0]
    raise KeyError(kind)


@pytest.mark.parametrize("kind", ["basic", "mixedrg", "gap", "highcov", "longspan", "capborder", "capgap", "capspill", "capfar",
                                  "wideins", "matepair", "longins", "overlap", "megadel", "manyrg"])
def test_packed_layout_reproduces_active_sets(kind, oracle_lib):
    from parity import run_oracle
    samples, params = _cohort(kind)
    headers = [[dict(name=rg.spec.name, median=rg.median, stddev=rg.stddev, read_length=rg.spec.read_length,
                     hist_start=rg.hist_start, hist_end=rg.hist_end, hist_counts=rg.hist_counts)
                for rg in s.read_groups] for s in samples]
    rgs = api.read_groups_from_headers(headers, params)
    sc = api.Scanner(params, rgs, len(samples), device=-1)        # host-only context
    anchor = api.cohort_anchor(samples)
    sc.begin_contig(anchor)
    g = 0
    for s in samples:
        for rg in s.read_groups:
            sc.push(g, rg.pos, rg.dev)
            g += 1
    n_windows = sc.window_count()
    _, _, n_ref, wins = run_oracle(samples, params, rgs, oracle_lib, window_sums=True, max_windows=n_windows + 10)
    assert n_windows == n_ref
    assert np.array_equal(wins[:, 0, 0], anchor + 30 * np.arange(n_ref))       # contiguous grid from the anchor
    for g in range(len(rgs)):
        got = sc.debug_host_window_sums(g, 0, n_windows)
        ref = wins[:, 1 + g, :]
        bad = np.nonzero((got != ref).any(axis=1))[0]
        assert bad.size == 0, f"rg {g}: first mismatch at window {bad[0]} (pos {anchor + 30 * bad[0]}): {got[bad[0]]} vs {ref[bad[0]]}"
    with pytest.raises(api.ScanError):
        sc.scan()                                                              # no CPU scan path
    sc.close()


def test_active_coverage_cap_equals_reference(oracle_lib):
    """ChromosomeProfile::add's stored / skipped decisions (profile_structure_popdel_call.h:1084-1113 with the lazily
    refreshed counter of getEndCount :870-928 and the zeroing of correctConsecutiveSwitch :722-737): the library's
    restatement (PdCapState, what pd_contig_push runs) and the oracle's, against what the reference's own ChromosomeProfile
    stored for the same streams (tests/golden/cap_replay.npz, made by make_golden.py with oracle/_ref/popdel_ref_harness)."""
    import ctypes as C
    import capcases
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "cap_replay.npz"))
    lib = api.load_library()
    u32p, u8p = C.POINTER(C.c_uint32), C.POINTER(C.c_uint8)
    for fn in (lib.pd_debug_cap_replay, oracle_lib.lib.orc_cap_replay):
        fn.restype, fn.argtypes = C.c_int, [C.c_uint32, C.c_uint32, C.c_uint64, u32p, u32p, u8p]
    dropped_by_stale_counter = 0
    for seed in capcases.SEEDS:
        max_load, start, end = capcases.cap_stream(seed)
        n, n_stored = (int(x) for x in gold[f"n{seed}"])
        assert n == start.size
        ref = np.unpackbits(gold[f"stored{seed}"])[:n]
        assert int(ref.sum()) == n_stored
        for name, fn in (("library", lib.pd_debug_cap_replay), ("oracle", oracle_lib.lib.orc_cap_replay)):
            got = np.zeros(n, dtype=np.uint8)
            assert fn(capcases.WINDOW_BUFFER, max_load, n, start.ctypes.data_as(u32p), end.ctypes.data_as(u32p), got.ctypes.data_as(u8p)) == 0
            bad = np.nonzero(got != ref)[0]
            assert bad.size == 0, f"{name}, seed {seed}: first difference at read pair {bad[0]} of {n} (start {start[bad[0]]})"
        # how often the reference's counter disagrees with the true number of open read pairs (round 1's rule)
        open_end, simple = [], np.zeros(n, dtype=np.uint8)
        for i in range(n):
            b = start[i] // 30
            open_end = [e for e in open_end if e >= b]
            if ref[i]:
                simple[i] = len(open_end) < max_load
                open_end.append(end[i] // 30)
            else:
                simple[i] = len(open_end) < max_load
        dropped_by_stale_counter += int((simple != ref).sum())
    assert dropped_by_stale_counter > 0          # the streams do exercise the lazy counter


def _tiny_scanner(device):
    samples, _ = simulate.simulate_cohort(seed=41, n_samples=2, contig_len=60_000, n_dels=0)
    params = api.CallParameters()
    rgs = api.read_groups_from_headers(api.cohort_headers(samples), params)
    return api.Scanner(params, rgs, len(samples), device=device), samples


def test_error_behaviour_of_the_c_abi_without_a_gpu():
    """Errors are return codes with a sticky message, never exceptions or exits; a host-only context (device = -1) packs
    and validates but refuses to scan -- there is no CPU fallback for the scan."""
    sc, samples = _tiny_scanner(device=-1)
    rg = samples[0].read_groups[0]
    with pytest.raises(api.ScanError, match="no open contig"):
        sc.push(0, rg.pos, rg.dev)
    sc2, _ = _tiny_scanner(device=-1)
    sc2.begin_contig(api.cohort_anchor(samples))
    with pytest.raises(api.ScanError, match="sorted"):
        sc2.push(0, rg.pos[::-1].copy(), rg.dev[::-1].copy())                  # PD_ERR_ORDER
    with pytest.raises(api.ScanError, match="sorted"):
        sc2.begin_contig(0)                                                     # sticky: the context stays failed
    sc3, _ = _tiny_scanner(device=-1)
    sc3.begin_contig(api.cohort_anchor(samples))
    sc3.push(0, rg.pos, rg.dev)
    sc3.reserve_windows(5000)
    assert sc3.window_count() > 1000
    with pytest.raises(api.ScanError, match="window_sums: host-only context"):
        sc3.debug_device_window_sums(0, 0, 100)                                # the device probe has no CPU path either
    with pytest.raises(api.ScanError, match="host-only context"):
        sc3.scan()
    sc4, _ = _tiny_scanner(device=-1)
    sc4.set_unify(50.0, 0.5, False)
    calls = np.zeros(2, dtype=api.CALL_DTYPE)
    with pytest.raises(api.ScanError, match=r"^\[-1\] pd_debug_unify: host-only context"):
        sc4.debug_unify(calls, np.zeros((2, 2, 13), np.uint32), 1)              # the merge probe has no CPU path: PD_ERR_ARG
    with pytest.raises(api.ScanError, match="no usable CUDA device|out of range"):
        _tiny_scanner(device=99)


def test_shard_attach_rejects_bad_arguments():
    import ctypes as C
    lib = api.load_library()
    sc, _ = _tiny_scanner(device=-1)
    mi = np.array([200, 200], dtype=np.uint32)
    spr = np.array([2, 2], dtype=np.uint32)
    info = api.PdShardInfo(0, 1, 4, 2, mi.ctypes.data_as(C.POINTER(C.c_uint32)), spr.ctypes.data_as(C.POINTER(C.c_uint32)))
    ctxs = (C.c_void_p * 2)(sc.ctx, sc.ctx)
    assert lib.pd_shard_attach_group(ctxs, 1, C.byref(info)) == -1             # PD_ERR_ARG: world < 2
    infos = (api.PdShardInfo * 2)(info, info)
    assert lib.pd_shard_attach_group(ctxs, 2, infos) != 0                       # infos[r].rank / world do not describe rank r of 2


def test_unify_staging_and_warmup_argument_checks():
    """pd_set_unify / pd_set_staging / pd_device_warmup: plain return codes, no GPU needed for the checks."""
    import ctypes as C
    lib = api.load_library()
    sc, _ = _tiny_scanner(device=-1)
    assert lib.pd_set_unify(None, None) == -1                                  # PD_ERR_ARG
    assert lib.pd_set_staging(None, 0) == -1
    sc.set_unify(50.0, 0.5, False)
    sc.set_unify(None)                                                         # back to window calls
    assert lib.pd_set_staging(sc.ctx, 0) == 0 and lib.pd_set_staging(sc.ctx, 1) == 0
    sc.set_staging(False)
    assert lib.pd_device_warmup(99) == -2                                      # PD_ERR_CUDA: no such device
    bad = api.PdUnifyParams(float("nan"), 0.5, 0, 0)
    assert lib.pd_set_unify(sc.ctx, C.byref(bad)) == -1
    with pytest.raises(api.ScanError, match="negative or NaN"):                # sticky
        sc.begin_contig(0)


def test_cli_dry_run_of_the_host_path(tmp_path):
    """`-g -1`: the shell's whole host path (profile decode, region handling, segment loader, host packer) without a scan:
    runs on a box without a GPU and writes a header-only VCF; option errors are reported, not crashed on."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cli = os.path.join(root, "popdel_b200", "popdel_b200_call")
    if not os.path.exists(cli):                                                # g++ only: links against the built scan library
        subprocess.run(["make", "-C", os.path.join(root, "popdel_b200", "host")], check=True, stdout=subprocess.DEVNULL)
    case = os.path.join(root, "tests", "golden", "twocontigs")
    out = tmp_path / "dry.vcf"
    r = subprocess.run([cli, "profiles.txt", "-g", "-1", "-o", str(out), "-r", "chrB:20001-60000", "-r", "chrA:50,001-100,000"],
                       cwd=case, capture_output=True, text=True, env=dict(os.environ, PD_TIMING="1"))
    assert r.returncode == 0, r.stderr
    assert "segments" in r.stderr and "decode" in r.stderr
    lines = open(out).read().splitlines()
    assert lines[0] == "##fileformat=VCFv4.3" and lines[-1].startswith("#CHROM") and lines[-1].endswith("sample00002")
    r = subprocess.run([cli, "profiles.txt", "-g", "-1", "-o", str(out), "-r", "chrZ:1-100"], cwd=case, capture_output=True, text=True)
    assert r.returncode != 0 and "Invalid chromosome name" in r.stderr
    r = subprocess.run([cli, "profiles.txt", "-g", "-1", "-o", str(out), "-A", "missing.txt"], cwd=case, capture_output=True, text=True)
    assert r.returncode != 0 and "coverage file" in r.stderr


@pytest.mark.parametrize("case,args", [("twocontigs", ["-r", "chrB:20001-60000", "-r", "chrA:50001-100000", "-R", "opt_rois.txt"]),
                                       ("gap", ["-r", "chr2:110001-790000"]), ("mixedrg", []), ("highcov", ["-x"])])
def test_cli_host_path_is_independent_of_the_thread_count(case, args, tmp_path):
    """The read pairs the shell hands to the scan (dry run, PD_DEBUG_DECODE checksums per read group and region) do not
    depend on how the decode is split: 1 thread, several tasks per file (index-offset cuts), more tasks than members."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cli = os.path.join(root, "popdel_b200", "popdel_b200_call")
    if not os.path.exists(cli):
        subprocess.run(["make", "-C", os.path.join(root, "popdel_b200", "host")], check=True, stdout=subprocess.DEVNULL)
    lst = "opt_x_profiles.txt" if "-x" in args else "profiles.txt"
    seen = []
    for threads in ("1", "7", "64"):
        r = subprocess.run([cli, lst, "-g", "-1", "-o", str(tmp_path / "dry.vcf")] + args, cwd=os.path.join(root, "tests", "golden", case),
                           capture_output=True, text=True, env=dict(os.environ, PD_DEBUG_DECODE="1", PD_THREADS=threads))
        assert r.returncode == 0, r.stderr
        seen.append([l for l in r.stderr.splitlines() if " pushed rg " in l])
    assert len(seen[0]) >= 3 and sum(int(l.split()[6]) for l in seen[0]) > 10000
    assert seen[0] == seen[1] == seen[2]


def test_cli_region_syntax_and_merging(tmp_path):
    """Region strings like the reference's parseGenomicRegion ("chr", "chr:begin", "chr:begin-end", thousands separators),
    -R files, sorting into the contig order of the first profile and merging of overlapping regions: equivalent
    spellings hand the same read pairs to the scan (dry run)."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cli = os.path.join(root, "popdel_b200", "popdel_b200_call")
    case = os.path.join(root, "tests", "golden", "twocontigs")

    def pushed(args):
        r = subprocess.run([cli, "profiles.txt", "-g", "-1", "-o", str(tmp_path / "dry.vcf")] + args, cwd=case, capture_output=True, text=True,
                           env=dict(os.environ, PD_DEBUG_DECODE="1"))
        assert r.returncode == 0, r.stderr
        return [l for l in r.stderr.splitlines() if " pushed rg " in l]

    rois = tmp_path / "rois.txt"
    rois.write_text("chrB:20,001-60,000\nchrA:50001-100000\n")
    a = pushed(["-r", "chrA:50001-100000", "-r", "chrB:20001-60000"])
    assert a == pushed(["-r", "chrB:20001-60000", "-r", "chrA:50001-100000"])            # contig order of the profile, not of the command line
    assert a == pushed(["-R", str(rois)])
    assert a == pushed(["-r", "chrA:50001-80000", "-r", "chrA:70001-100000", "-R", str(rois)])   # overlapping regions are merged
    assert len(a) == 6                                                                   # 2 regions x 3 read groups
    whole = pushed([])
    assert whole == pushed(["-r", "chrA", "-r", "chrB", "-r", "chrC"]) == pushed(["-r", "chrA:1", "-r", "chrB"])
    assert pushed(["-r", "chrC"]) == []                                                  # a contig without read pairs
    r = subprocess.run([cli, "profiles.txt", "-g", "-1", "-o", str(tmp_path / "dry.vcf"), "-r", "chrA:12x-40"], cwd=case, capture_output=True, text=True)
    assert r.returncode != 0 and "parsing genomic region" in r.stderr


def test_cli_rejects_truncated_and_empty_inputs(tmp_path):
    """A profile cut off inside a gzip member must stop the shell (it used to lose read pairs silently), and so must an
    empty profile list (dry run: -g -1 needs no GPU)."""
    import subprocess
    cli = os.path.join(ROOT, "popdel_b200", "popdel_b200_call")
    src = os.path.join(ROOT, "tests", "golden", "basic", "sample00000.profile")
    data = open(src, "rb").read()
    cut = tmp_path / "cut.profile"
    cut.write_bytes(data[:len(data) // 2])
    lst = tmp_path / "list.txt"
    lst.write_text(str(cut) + "\n")
    r = subprocess.run([cli, str(lst), "-g", "-1", "-o", str(tmp_path / "x.vcf")], capture_output=True, text=True)
    assert r.returncode != 0 and "truncated" in r.stderr
    lst.write_text("\n")
    r = subprocess.run([cli, str(lst), "-g", "-1", "-o", str(tmp_path / "x.vcf")], capture_output=True, text=True)
    assert r.returncode != 0 and "no profiles" in r.stderr
