#!/usr/bin/env python
"""bench.py -- `popdel call` window scan throughput (sample x window genotype evaluations per second).

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --steps K --dump-outputs bench_outputs    (also writes the last timed step's results as bench_outputs/*.npy)

Workload (BASELINE.json configs[1]): 100 synthetic profiles, chr21 (46,709,983 bp -> 1.56e6 windows of 30 bp), one
read group each (30x, 2x150 bp, insert ~ N(500, 50^2)), planted deletions; per GPU one such window range (weak
scaling over contiguous window ranges, no data-path collective). A step = one pass of the scan over the range.
  value : evaluations/s with the packed read pairs already resident in HBM: all kernels of the scan incl. the
          segment-level merge on the device (pd_set_unify, the product's default: `popdel call` writes merged variants)
          + result copy-back; `other_output` = the same returning every window call with its per-sample row (50 MB
          per chr21 step over PCIe)
  e2e   : evaluations/s through the C ABI from host arrays: push + H2D + device packing + scan + D2H
  roofline : the WHOLE scan: SURVEY.md 8d's 20 B per evaluation x evaluations per step / device time of a step
             (CUDA events on the library's stream); `k_stream` = the HBM-bound screen kernel on its own
  parity_check : the calls of the first --cpu-slice bp compared with the CPU oracle (integers exact, LR / AF 1e-6)
  cpu_baseline : the CPU oracle port (1 core) on a bounded slice of the same cohort
The reference arm times the reference's own `popdel call` (oracle/_ref/popdel_ref, built from /root/reference by
oracle/Makefile) on profile files of a bounded slice of the same workload, one process per host core over contiguous
regions (-r), like BASELINE.md section 3.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CHR21_LEN = 46_709_983
METRIC = "sample x window genotype evaluations per second (popdel call window scan)"
UNIT = "evals/s"


# ----------------------------------------------------------------------------------------------------------------
# synthetic cohort (host arrays)
# ----------------------------------------------------------------------------------------------------------------
def plant(seed, n_samples, length, per_mbp):
    rng = np.random.default_rng([seed, 911])
    n = max(1, int(round(length / 1e6 * per_mbp)))
    slot = (length - 40_000) // n
    starts, lens, gts = [], [], []
    for k in range(n):
        L = int(np.exp(rng.uniform(np.log(300), np.log(10000))))
        s = 20_000 + k * slot + int(rng.integers(0, max(1, slot - L - 2000)))
        af = float(rng.choice([0.1, 0.3, 0.5]))
        g = rng.binomial(2, af, size=n_samples).astype(np.uint8)
        if g.sum() == 0:
            g[int(rng.integers(0, n_samples))] = 1
        starts.append(s), lens.append(L), gts.append(g)
    return np.array(starts, np.uint32), np.array(lens, np.uint32), np.stack(gts)


def cohort_specs(seed, n_samples, mixed=False):
    """(sample, read group, mu, sigma, read pairs per bp) of every read group of the cohort."""
    rng = np.random.default_rng([seed, 77])
    specs = []
    for s in range(n_samples):
        k = int(rng.integers(1, 4)) if mixed else 1
        for j in range(k):
            mu = float(rng.choice([350, 450, 550])) if mixed else 500.0
            sd = float(rng.choice([30, 50, 80])) if mixed else 50.0
            specs.append((s, len(specs), mu, sd, 0.1 / k))
    return specs


def make_cohort(seed, n_samples, length, per_mbp, threads, mixed=False, sample_range=None, gen_length=None):
    """Returns (list of read groups [pos, isize, dev, header, sample], deletions). One read group per sample, or with
    `mixed` 1-3 read groups per sample with mu in {350,450,550} and sigma in {30,50,80} (BASELINE.json configs[2]).
    sample_range = (s0, s1): only the read groups of these samples of the cohort are generated (sample sharding)."""
    from popdel_b200 import api
    ds, dl, gt = plant(seed, n_samples, length, per_mbp)
    specs = cohort_specs(seed, n_samples, mixed)
    if sample_range is not None:
        specs = [sp for sp in specs if sample_range[0] <= sp[0] < sample_range[1]]

    glen = length if gen_length is None else gen_length        # (deletions are planted for `length`; only [0, glen) is generated)
    near = ds < glen + 40_000

    def one(spec):
        s, g, mu, sd, dens = spec
        pos, isz = api.synth_read_group(seed, g, mu, sd, 150, dens, 0, glen, ds[near], dl[near], gt[near, s])
        med = int(mu)
        lo, hi = max(1, int(np.floor(med - 3 * sd))), int(np.ceil(med + 3 * sd)) + 1
        sel = isz[(isz >= lo) & (isz < hi)]
        counts = np.bincount(sel - lo, minlength=hi - lo).astype(np.float64)
        hdr = dict(name=f"rg{g}", median=med, stddev=sd, read_length=150, hist_start=lo, hist_end=hi, hist_counts=counts)
        dev = isz - np.int32(med)
        return pos, isz, dev, hdr, s

    with ThreadPoolExecutor(threads) as ex:
        out = list(ex.map(one, specs))
    return out, (ds, dl, gt)


def workload_config(N, L, mixed, dels_per_mbp, world):
    """`config` of the JSON line: the same for both arms (the reference arm times a bounded sample of this workload and says
    so in cpu_baseline.sample)."""
    return {"workload": f"{N} synthetic profiles x chr21-sized window range ({L} bp, {L // 30} windows of 30 bp) per GPU, "
                        f"{'1-3 read groups per sample with mixed insert-size histograms' if mixed else 'single read group each'}, "
                        f"30x, planted deletions {dels_per_mbp}/Mbp; inputs larger than the 126 MB L2",
            "samples": N,
            "parallelism": f"window-range x{world} (one range per GPU, same synthetic content in every range, no data-path collective)"}


def write_profiles(cohort, N, tmp, cores):
    from popdel_b200 import profile_format as pf
    contigs = [("chr21", CHR21_LEN)]

    def write(s):
        p = os.path.join(tmp, f"s{s:05d}.profile")
        pf.write_profile_single_rg(p, cohort[s][3], contigs, 0, cohort[s][0], cohort[s][1], compressed=True)
        return p

    with ThreadPoolExecutor(cores) as ex:
        paths = list(ex.map(write, range(N)))
    lst = os.path.join(tmp, "profiles.txt")
    open(lst, "w").write("\n".join(paths) + "\n")
    return paths, lst


def run_reference_regions(binary, lst, tmp, slice_bp, cores):
    """The unmodified reference binary, one process per core over contiguous -r regions; returns the wall time."""
    regions = np.linspace(0, slice_bp, cores + 1).astype(int)
    t0 = time.perf_counter()
    procs = [subprocess.Popen([binary, "call", lst, "-r", f"chr21:{regions[i] + 1}-{regions[i + 1]}", "-o",
                               os.path.join(tmp, f"out{i}.vcf")], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
             for i in range(cores)]
    rc = [p.wait() for p in procs]
    assert all(r == 0 for r in rc), rc
    return time.perf_counter() - t0


def e2e_files(args):
    """Same files in, VCF out: the drop-in shell popdel_b200_call against the unmodified reference binary on the SAME gzip
    profiles of a bounded slice of the workload (what scripts/cli_bench.py does)."""
    binary = os.path.join(ROOT, "oracle", "_ref", "popdel_ref")
    ours = os.path.join(ROOT, "popdel_b200", "popdel_b200_call")
    if not (os.path.exists(binary) and os.path.exists(ours)):
        return {"unavailable": "oracle/_ref/popdel_ref or popdel_b200/popdel_b200_call not built"}
    cores = os.cpu_count() or 1
    N = args.samples
    slice_bp = int(min(args.ref_slice, args.length))
    cohort, _ = make_cohort(args.seed, N, slice_bp, args.dels_per_mbp, cores)
    tmp = tempfile.mkdtemp(prefix="popdel_e2e_files_")
    try:
        paths, lst = write_profiles(cohort, N, tmp, cores)
        walls = []
        for _ in range(2):                       # cold, warm
            t0 = time.perf_counter()
            r = subprocess.run([ours, lst, "-o", os.path.join(tmp, "ours.vcf")], capture_output=True, text=True)
            walls.append(time.perf_counter() - t0)
            assert r.returncode == 0, r.stderr
        t_ref = run_reference_regions(binary, lst, tmp, slice_bp, cores)
        evals = N * (slice_bp // 30)
        return {"slice_bp": slice_bp, "profile_bytes": int(sum(os.path.getsize(p) for p in paths)), "host_cores": cores,
                "ours_s": walls[-1], "ours_cold_s": walls[0], "reference_s": t_ref, "ours_evals_per_s": evals / walls[-1],
                "reference_evals_per_s": evals / t_ref, "speedup": t_ref / walls[-1],
                "note": "gzip profile files -> VCF: popdel_b200_call (1 GPU + host cores for the decode) vs the unmodified reference, "
                        "one process per host core over -r regions"}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def bind_to_gpu_numa_node(local_rank):
    """Runs this rank (and therefore its page-locked buffers, first-touch) on the CPUs of the NUMA node its GPU hangs off:
    at 8 ranks per box the host->device copies of the e2e step otherwise cross the socket interconnect. Best effort."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        if hasattr(pr, "pci_bus_id") and hasattr(pr, "pci_device_id"):
            bus = "%04x:%02x:%02x.0" % (getattr(pr, "pci_domain_id", 0), pr.pci_bus_id, pr.pci_device_id)
        else:
            out = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                                 capture_output=True, text=True, timeout=20).stdout.strip().lower()
            bus = out[4:] if len(out.split(":")[0]) == 8 else out          # 00000000:1b:00.0 -> 0000:1b:00.0
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return {"node": node, "cpus": len(allowed)}
    except Exception:
        pass
    return None


class ClockSampler:
    def __init__(self, dev):
        self.dev, self.proc, self.lines = dev, None, []

    def start(self):
        if self.dev is None:                     # only rank 0 polls the driver (every rank doing so perturbs the timed steps)
            return
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.dev), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True).start()
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=[])
        t_end = time.time() + 5.0                # nvidia-smi can take longer to start than a short timed region lasts
        while not self.lines and time.time() < t_end and self.proc.poll() is None:
            time.sleep(0.05)
        time.sleep(0.05)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            t = [x.strip() for x in ln.split(",")]
            if len(t) < 6:
                continue
            try:
                sm.append(float(t[0])), (mx := float(t[1]))
            except ValueError:
                continue
            for nm, v in zip(names, t[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=mx, reasons=sorted(reasons))


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


DUMP_BYTES = 64 << 20


def output_arrays(res, budget=DUMP_BYTES):
    """What a caller of Scanner.scan() receives, as float64 arrays (exact for every field): each field of the calls, the
    per-sample rows and, with the device-side merge, the significant-window counts. Beyond `budget` bytes a fixed, seeded
    sample of the calls is kept; `call_index` says which. Copies: a scan(copy=False) result is overwritten by the next scan."""
    calls, per, sig = res["calls"], res["per_sample"], res["significant_windows"]
    n = len(calls)
    row_bytes = 8 * (len(calls.dtype.names) + per[0].size + (sig is not None) + 1) if n else 8
    rows = np.arange(n)
    if n * row_bytes > budget - 4096:                                   # (4 kB for the .npy headers and the counts)
        k = max(0, (budget - 4096) // row_bytes)
        rows = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
    out = {f"calls_{f}": calls[f][rows] for f in calls.dtype.names}
    out["per_sample"] = per[rows]
    if sig is not None:
        out["significant_windows"] = sig[rows]
    out["call_index"] = rows
    out["n_calls"] = np.array([n])
    out["n_windows"] = np.array([res["n_windows"]])
    out["n_window_calls"] = np.array([res["n_window_calls"]])
    return {k: np.asarray(v, dtype=np.float64) for k, v in out.items()}


def write_outputs(d, arrays):
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, f"{name}.npy"), a)


# ----------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch
    from popdel_b200 import api, sharding
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    threads = max(1, min(len(os.sched_getaffinity(0)), (os.cpu_count() or 8) // max(world, 1)))
    N, L = args.samples, args.length
    t0 = time.time()
    # weak scaling over window ranges: every rank scans its own range; the ranges get the SAME synthetic content so that
    # the per-rank work is identical and the N-GPU value measures scaling, not the luck of the planted deletions
    cohort, dels = make_cohort(args.seed, N, L, args.dels_per_mbp, threads, args.mixed)
    t_gen = time.time() - t0
    params = api.CallParameters()
    rgs = api.read_groups_from_headers([[c[3] for c in cohort if c[4] == s] for s in range(N)], params)
    R = len(cohort)
    sc = api.Scanner(params, rgs, N, device=local_rank)
    anchor = (min(int(c[0][0]) for c in cohort) // 30) * 30

    def push_all():
        sc.begin_contig(anchor)
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(lambda g: sc.push(g, cohort[g][0], cohort[g][2]), range(R)))

    # page-locked copies of the host arrays for the end-to-end path (pd_contig_push_pinned packs on the device)
    def pin(a):
        t = torch.from_numpy(a.view(np.int32)).pin_memory()
        return t, t.numpy().view(a.dtype)
    pinned = [(pin(np.ascontiguousarray(c[0], dtype=np.uint32)), pin(np.ascontiguousarray(c[2], dtype=np.int32))) for c in cohort]

    def push_all_pinned():
        sc.begin_contig(anchor)
        for g in range(R):
            sc.push_pinned(g, pinned[g][0][1], pinned[g][1][1])

    # the same read pairs in the 4-byte form of pd_contig_push_compact32 (what a profile decoder emits directly: the file stores
    # a u8 offset per 256-bp window and an i32 deviation), page-locked; and in round 2's earlier 5-byte form (65 536-bp blocks)
    def pin_any(a, dt):
        t = torch.from_numpy(a.view(dt)).pin_memory()
        return t, t.numpy().view(a.dtype)
    compact, compact5 = [], []
    for c in cohort:
        w32, blk8 = api.compact32_encode(c[0], c[2])
        compact.append((pin_any(w32, np.int32), pin_any(blk8, np.int32)))
        if world == 1:                                              # (the 5-byte leg is an N=1 side measurement: 2.3 GB of pinned memory per rank)
            lo, d24, blk = api.compact_encode(c[0], c[2])
            compact5.append((pin_any(lo, np.int16), pin_any(d24, np.uint8), pin_any(blk, np.int32)))

    def push_all_compact():
        sc.begin_contig(anchor)
        for g in range(R):
            sc.push_compact32(g, compact[g][0][1], compact[g][1][1])

    def push_all_compact5():
        sc.begin_contig(anchor)
        for g in range(R):
            sc.push_compact(g, compact5[g][0][1], compact5[g][1][1], compact5[g][2][1])

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident-input throughput. --output unify (default, the product's default: `popdel call` writes merged variants): the
    # segment-level merge runs on the device (pd_set_unify), only merged variants cross PCIe; --output calls: every window call
    # of every processSegment() with its per-sample row (the reference's String<Call> before unifyCalls) is copied back --
    # 50 MB per chr21 step, 11 % faster on one GPU but 8 GPUs then push 80 GB/s into one host (measured r02: 67 % of linear
    # at N=8 against 98 % with the merge on the device). The other mode is timed as well (fewer steps) and reported beside it.
    push_all()
    sc.upload()
    mean_sd = float(np.mean([r.as_dict()["stddev"] for r in rgs]))
    res_w = sc.scan(copy=True)                    # window calls (parity leg, counts)
    evals = int(res_w["n_windows"]) * N
    main_unify = args.output == "unify"

    def set_mode(unify_on):
        if unify_on:
            sc.set_unify(mean_sd, 0.5, False)
        else:
            sc.set_unify(None)

    set_mode(main_unify)
    res = sc.scan(copy=False)
    clocks = ClockSampler(local_rank if rank == 0 else None)      # started before the warm-up steps so that it is sampling when the timed steps run
    clocks.start()
    for _ in range(args.warmup):
        res = sc.scan(copy=False)
    t_w = time.time()
    while clocks.proc and not clocks.lines and time.time() - t_w < 5.0:     # more untimed warm-up steps until nvidia-smi delivers samples
        res = sc.scan(copy=False)
    barrier()
    t0 = time.perf_counter()
    ms_screen, ms_dev, ms_scr_all, ms_gen, ms_em, launches = [], [], [], [], [], 0
    for _ in range(args.steps):
        res = sc.scan(copy=False)
        ms_screen.append(res["ms_stream"]), ms_dev.append(res["ms_total"]), ms_scr_all.append(res["ms_screen"]), ms_gen.append(res["ms_genotype"])
        ms_em.append(res["ms_em"])
        launches += int(res["n_kernel_launches"])
    barrier()
    dt = time.perf_counter() - t0
    dumped = output_arrays(res) if args.dump_outputs and rank == 0 else None
    n_lines = len(clocks.lines)
    t_w = time.time()
    while clocks.proc and len(clocks.lines) == n_lines and time.time() - t_w < 1.0:   # keep the load up until the sampler has seen it
        sc.scan(copy=False)
    clk = clocks.stop()
    dt, evals_all = sharding.reduce_timing(dt, float(evals), dist, "cuda")      # max over ranks / sum over ranks
    value = evals_all * args.steps / dt
    n_out, d2h_main, n_wcalls = int(len(res["calls"])), int(res["d2h_bytes"]), int(res["n_window_calls"])

    # ---- the other output mode
    set_mode(not main_unify)
    ro = sc.scan(copy=False)
    barrier()
    t0 = time.perf_counter()
    o_steps = max(1, min(args.steps, 5))
    ms_dev_o, ms_uni = [], []
    for _ in range(o_steps):
        ro = sc.scan(copy=False)
        ms_dev_o.append(ro["ms_total"]), ms_uni.append(ro["ms_unify"])
    barrier()
    dto = time.perf_counter() - t0
    dto, _ = sharding.reduce_timing(dto, float(evals), dist, "cuda")
    other = {"output": "calls" if main_unify else "unify", "value": evals_all * o_steps / dto, "ms_per_step": dto / o_steps * 1e3,
             "ms_device_per_step": float(np.mean(ms_dev_o)), "records": int(len(ro["calls"])), "d2h_bytes_per_step": int(ro["d2h_bytes"])}
    if not main_unify:
        other["ms_unify_kernels"] = float(np.mean(ms_uni))
        other["note"] = "pd_set_unify: window calls and their per-sample rows stay in device memory, every segment is merged there (unifyCalls)"
    n_variants = int(len(ro["calls"])) if not main_unify else n_out

    # ---- end to end through the C ABI from host arrays (pack -> pinned -> H2D -> scan -> D2H)
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    set_mode(main_unify)
    push_all_compact()
    r2 = sc.scan(copy=False)                                        # warm-up (device buffers exist afterwards)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        push_all_compact()
        r2 = sc.scan(copy=False)
    barrier()
    dt2 = time.perf_counter() - t0
    dt2, _ = sharding.reduce_timing(dt2, float(evals), dist, "cuda")
    e2e = evals_all * e2e_steps / dt2
    assert len(r2["calls"]) == n_out, (len(r2["calls"]), n_out)
    # the same in the 5-byte form (N=1 only)
    five = None
    if world == 1:
        push_all_compact5()
        r25 = sc.scan(copy=False)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            push_all_compact5()
            r25 = sc.scan(copy=False)
        dt25 = time.perf_counter() - t0
        assert len(r25["calls"]) == n_out
        five = {"value": evals_all * e2e_steps / dt25, "ms_per_step": dt25 / e2e_steps * 1e3, "h2d_bytes_per_step": int(r25["h2d_bytes"]),
                "path": "pd_contig_push_compact: 16-bit position remainders per 65 536-bp block + 24-bit deviations"}
    # the same from raw page-locked pos[] / dev[] arrays (8 bytes per read pair)
    push_all_pinned()
    r2r = sc.scan(copy=False)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        push_all_pinned()
        r2r = sc.scan(copy=False)
    barrier()
    dt2r = time.perf_counter() - t0
    dt2r, _ = sharding.reduce_timing(dt2r, float(evals), dist, "cuda")
    assert len(r2r["calls"]) == n_out
    # PCIe floor of that path: the same page-locked arrays copied to the device with nothing else going on
    dev_bufs = [(torch.empty_like(p[0][0], device="cuda"), torch.empty_like(p[1][0], device="cuda")) for p in pinned]
    for _ in range(2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for (pp, dd), (dp, ddv) in zip(pinned, dev_bufs):
            dp.copy_(pp[0], non_blocking=True), ddv.copy_(dd[0], non_blocking=True)
        torch.cuda.synchronize()
        dt_copy = time.perf_counter() - t0
    raw_bytes = sum(p[0][0].numel() * 4 + p[1][0].numel() * 4 for p in pinned)
    del dev_bufs
    dev_bufs = [tuple(torch.empty_like(q[0], device="cuda") for q in cq) for cq in compact]
    for _ in range(2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for cq, db in zip(compact, dev_bufs):
            for q, d_ in zip(cq, db):
                d_.copy_(q[0], non_blocking=True)
        torch.cuda.synchronize()
        dt_copy_c = time.perf_counter() - t0
    compact_bytes = sum(sum(q[0].numel() * q[0].element_size() for q in cq) for cq in compact)
    del dev_bufs
    # the same through pd_contig_push (sequential host packer, one thread per read group)
    push_all()
    r3 = sc.scan(copy=False)
    barrier()
    t0 = time.perf_counter()
    push_all()
    r3 = sc.scan(copy=False)
    barrier()
    dt3 = time.perf_counter() - t0
    dt3, _ = sharding.reduce_timing(dt3, float(evals), dist, "cuda")

    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    peak, peak_src = measured_peak_gbs()
    ms_s = float(np.mean(ms_screen))
    ms_d = float(np.mean(ms_dev))
    default_wl = N == 100 and L == CHR21_LEN and args.seed == 1 and not args.mixed and abs(args.dels_per_mbp - 2.0) < 1e-9
    traffic = None                      # DRAM bytes of one launch / one scan from the committed ncu --set full captures (default workload only)
    tpath = os.path.join(ROOT, "profiles", "r02", "traffic.json")
    tj = json.load(open(tpath)) if os.path.exists(tpath) and default_wl else {}
    fused = R == N and N <= 256
    algo_bytes = 20 * evals             # SURVEY.md 8d: rho * 4 B + 8 B = 20 B per evaluation at 30x (the design moves 12: 4 B per read pair)
    achieved = algo_bytes / (ms_d * 1e-3) / 1e9
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32 (screen) / f64 (likelihoods)", "data": "synthetic",
        "config": workload_config(N, L, args.mixed, args.dels_per_mbp, world),
        "workload_detail": {"read_groups": R, "windows_per_gpu": int(res["n_windows"]), "read_pairs_per_gpu": int(res["n_reads"]),
                            "packed_bytes": int(res["algorithmic_bytes"]),
                            "output": "merged variants per segment (unifyCalls on the device, pd_set_unify)" if main_unify else
                                      "window calls of every processSegment() + per-sample rows (pd_contig_scan's own product)",
                            "calls_per_step": n_wcalls, "variants_per_step": n_variants, "d2h_bytes_per_step": d2h_main,
                            "flagged_windows": int(res["n_flagged_windows"]), "candidates": int(res["n_candidates"])},
        "clocks": clk,
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(r2["h2d_bytes"]), "d2h_bytes_per_step": int(r2["d2h_bytes"]),
                "steps": e2e_steps, "ms_per_step": dt2 / e2e_steps * 1e3, "path": "pd_contig_push_compact32 (4 B per read pair + 4 B per 256-bp block over PCIe, expansion + packing on the device) + pd_contig_scan" + (" with pd_set_unify" if main_unify else ""),
                "pcie": {"h2d_gbs_plain_copy": compact_bytes / dt_copy_c / 1e9, "floor_ms_per_step": dt_copy_c * 1e3,
                         "frac_of_floor": dt_copy_c / (dt2 / e2e_steps),
                         "note": "floor = the same page-locked arrays copied host->device with nothing else running; "
                                 "the e2e step additionally expands and packs on the device, scans and writes the results back"},
                "five_byte_form": five,
                "raw_arrays": {"value": evals_all * e2e_steps / dt2r, "ms_per_step": dt2r / e2e_steps * 1e3, "h2d_bytes_per_step": int(r2r["h2d_bytes"]),
                               "floor_ms_per_step": dt_copy * 1e3, "path": "pd_contig_push_pinned: raw pos[] / dev[] arrays, 8 B per read pair"},
                "host_packer_value": evals_all / dt3, "host_packer_ms_per_step": dt3 * 1e3, "host_packer_h2d_bytes": int(r3["h2d_bytes"])},
        "gpu_launches": launches,
        "other_output": other,
        "roofline": {"bound": "hbm", "kernel": "scan (all kernels of a step)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": tj.get("scan", {}).get("dram_bytes_per_step"),
                     "peak_source": peak_src, "bytes_per_eval": 20, "algorithmic_bytes_per_launch": int(algo_bytes),
                     "ms_device_per_step": ms_d, "ms_screen": float(np.mean(ms_scr_all)), "ms_genotype": float(np.mean(ms_gen)),
                     "frac_at_own_bytes": res["algorithmic_bytes"] / (ms_d * 1e-3) / 1e9 / peak,
                     "own_bytes_per_eval": res["algorithmic_bytes"] / evals,
                     "k_stream": {"achieved": res["algorithmic_bytes"] / (ms_s * 1e-3) / 1e9, "frac": res["algorithmic_bytes"] / (ms_s * 1e-3) / 1e9 / peak,
                                  "ms_kernel": ms_s, "share_of_step": ms_s / ms_d, "algorithmic_bytes_per_launch": int(res["algorithmic_bytes"]),
                                  "traffic": tj.get("k_stream", {}).get("dram_bytes_per_launch"),
                                  "note": "the only HBM-bound kernel: every packed read-pair word (4 B) once, read-only"},
                     "dominant_kernel_by_time": {
                         "kernel": "k_em_one" if fused else "k_e2_* (pd_em2.cu)", "ms": float(np.mean(ms_em)),
                         "pairs_timed": int(res["n_em_pairs_timed"]), "pairs_per_step": int(res["n_candidates"]),
                         "share_of_step": float(np.mean(ms_em)) / ms_d if int(res["n_em_pairs_timed"]) == int(res["n_candidates"]) else None,
                         "bound": "L1TEX / LSU wavefronts of the likelihood-table gathers + fp64; not HBM, not tensor (profiles/r02)"},
                     "note": "achieved = SURVEY.md 8d's algorithmic bytes (20 B per sample x window evaluation) / device time of one step "
                             "(CUDA events on the library's stream around ALL kernels of the scan incl. the device-side merge)"},
        "setup_s": {"generate": t_gen}, "numa_binding_rank0": numa,
    }
    if world == 1 and not args.no_cpu_baseline:
        base, ref_calls, ref_ps = cpu_baseline(args, cohort, params, rgs)
        out["cpu_baseline"] = base
        # parity leg: the window calls of the GPU scan inside the oracle's slice (minus the longest read-pair span at its end,
        # where the oracle saw no read pairs beyond the slice) must equal the oracle's
        lim = int(args.cpu_slice) - 25_000
        gsel = res_w["calls"]["window_position"] < lim
        osel = ref_calls["window_position"] < lim
        from parity import assert_calls_equal
        assert_calls_equal(res_w["calls"][gsel], res_w["per_sample"][gsel], ref_calls[osel], ref_ps[osel])
        out["parity_check"] = (f"{int(osel.sum())} window calls == CPU oracle (windows below {lim} bp: integers and per-sample "
                               f"PL/LAD/DAD/FL bit-exact, LR / AF within 1e-6 relative)")
    if world == 1 and not args.no_e2e_files:
        # the command-line tool is a process of its own: give the GPU and the page-locked host memory back first (its CUDA
        # start-up was measured between 0.3 and 4 s while this process still held its context and 8 GB of pinned buffers)
        sc.close()
        sc._pinned_keep = {}
        pinned.clear(); compact.clear(); compact5.clear()
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        out["e2e_files"] = e2e_files(args)
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    emit_json(out)


def cpu_baseline(args, cohort, params, rgs):
    """The CPU oracle (restatement of the reference, 1 core) on the first `slice` bp of the same cohort."""
    import oracle_api
    so = os.path.join(ROOT, "oracle", "liboracle.so")
    if not os.path.exists(so):
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "oracle"], check=True, stdout=subprocess.DEVNULL)
    orc = oracle_api.load(so)
    N = args.samples
    slice_bp = int(args.cpu_slice)
    pos, dev, off = [], [], [0]
    for c in cohort:
        n = int(np.searchsorted(c[0], slice_bp))
        pos.append(c[0][:n]), dev.append(c[2][:n]), off.append(off[-1] + n)
    t0 = time.perf_counter()
    calls, ps, nwin = orc.scan_contig(params.as_dict(), [r.as_dict() for r in rgs], np.array(off, np.uint64),
                                      np.concatenate(pos), np.concatenate(dev), N, max_calls=200000)
    dt = time.perf_counter() - t0
    return ({"value": nwin * N / dt, "unit": UNIT, "cores": 1, "kind": "port",
             "sample": f"first {slice_bp} bp of the same cohort: {nwin} windows x {N} samples in {dt:.1f} s ({len(calls)} window calls)"},
            calls, ps)


# ----------------------------------------------------------------------------------------------------------------
# sample-sharded cohort (BASELINE.json configs[4] style): every rank holds samples/world samples of the SAME window range
# ----------------------------------------------------------------------------------------------------------------
def run_sample_sharded(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from popdel_b200 import api
    assert world >= 2, "--shard-samples needs torchrun with >= 2 ranks"
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    threads = max(1, (os.cpu_count() or 8) // world)
    N, L = args.samples, args.length
    spr = api.split_samples(N, world)
    s0 = sum(spr[:rank])
    # with --device-gen the host generator only makes a short sample per read group for the histograms of the headers
    hdr_len = min(L, 300_000) if args.device_gen else L
    cohort, dels = make_cohort(args.seed, N, L, args.dels_per_mbp, threads, args.mixed, sample_range=(s0, s0 + spr[rank]), gen_length=hdr_len)
    params = api.CallParameters()
    # call parameters of the WHOLE cohort (only sigma of the other ranks' read groups is needed)
    specs = cohort_specs(args.seed, N, args.mixed)
    every = [api.ReadGroup(sample=sp[0], median=int(sp[2]), read_length=150, stddev=sp[3], offset=0, values=np.zeros(3), min_prob=0.0,
                           lower_quantile_dist=0, upper_quantile_dist=0) for sp in specs]
    params.finalize(every)
    min_init = np.array([r.min_init_del_len for r in every], dtype=np.uint32)
    p_local = api.CallParameters(min_len=params.min_len)
    rgs = api.read_groups_from_headers([[c[3] for c in cohort if c[4] == s] for s in range(s0, s0 + spr[rank])], p_local)
    assert [r.min_init_del_len for r in rgs] == [int(min_init[sp[1]]) for sp in specs if s0 <= sp[0] < s0 + spr[rank]]
    uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        uid.copy_(torch.frombuffer(bytearray(api.shard_unique_id()), dtype=torch.uint8))
    dist.broadcast(uid, 0)
    sc = api.Scanner(params, rgs, spr[rank], device=local_rank)
    sc.attach_nccl(rank, world, spr, min_init, bytes(uid.cpu().numpy()))
    sc.begin_contig(0)
    sc.reserve_windows(L // 30 + 2)
    if args.device_gen:
        assert not args.check, "--check compares with the CPU oracle on host arrays"
        ds, dl, gt = dels
        local = [(sp[0] - s0,) + tuple(sp[1:]) for sp in specs if s0 <= sp[0] < s0 + spr[rank]]
        gen = api.SynthDevice(local_rank)
        _, dp, dd, rs = gen.generate(args.seed, local, 0, L, ds, dl, np.ascontiguousarray(gt[:, s0:s0 + spr[rank]]), spr[rank])
        for g in range(len(local)):
            sc.push_device(g, int(rs[g + 1] - rs[g]), dp + 4 * int(rs[g]), dd + 4 * int(rs[g]))
    else:
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(lambda g: sc.push(g, cohort[g][0], cohort[g][2]), range(len(cohort))))
    sc.upload()
    res = sc.scan(copy=True)
    evals = int(res["n_windows"]) * N
    check = None
    if args.check:                      # merged result against the CPU oracle (small cohorts only)
        parts = [None] * world
        dist.all_gather_object(parts, dict(calls=res["calls"], per_sample=res["per_sample"], pos=[c[0] for c in cohort], dev=[c[2] for c in cohort],
                                           rgs=[r.as_dict() for r in rgs]))
        if rank == 0:
            import oracle_api
            from parity import assert_calls_equal
            orc = oracle_api.load(os.path.join(ROOT, "oracle", "liboracle.so"))
            for p in parts[1:]:
                assert np.array_equal(p["calls"], parts[0]["calls"]), "ranks disagree on the calls"
            per = np.concatenate([p["per_sample"] for p in parts], axis=1)
            pos = [a for p in parts for a in p["pos"]]
            dev = [a for p in parts for a in p["dev"]]
            rg_all, base = [], 0
            for r, p in enumerate(parts):
                for d in p["rgs"]:
                    rg_all.append({**d, "sample": d["sample"] + base})
                base += spr[r]
            off = np.concatenate([[0], np.cumsum([a.size for a in pos])]).astype(np.uint64)
            ref_calls, ref_ps, nwin = orc.scan_contig(params.as_dict(), rg_all, off, np.concatenate(pos), np.concatenate(dev), N, max_calls=400000)
            assert nwin == res["n_windows"], (nwin, res["n_windows"])
            assert_calls_equal(parts[0]["calls"], per, ref_calls, ref_ps)
            check = f"merged calls of {world} ranks == CPU oracle ({len(ref_calls)} window calls, integers bit-exact, LR/AF 1e-6)"
    for _ in range(args.warmup):
        sc.scan(copy=False)
    clocks = ClockSampler(local_rank)
    clocks.start()
    dist.barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    launches, ms_dev = 0, []
    for _ in range(args.steps):
        r2 = sc.scan(copy=False)
        launches += int(r2["n_kernel_launches"]); ms_dev.append(r2["ms_total"])
    dist.barrier(); torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    clk = clocks.stop()
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t.item())
    n_calls = len(r2["calls"])
    sc.close()
    dist.barrier()
    dist.destroy_process_group()
    if rank != 0:
        return
    out = {"metric": METRIC, "value": evals * args.steps / dt, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "int32 (screen) / f64 (likelihoods)", "data": "synthetic",
           "config": {"workload": f"{N} synthetic profiles sharded BY SAMPLE over {world} GPUs ({spr[0]} per GPU), one window range of {L} bp "
                                  f"({res['n_windows']} windows), {'mixed read groups' if args.mixed else 'single read group each'}, 30x, "
                                  f"planted deletions {args.dels_per_mbp}/Mbp; exchanges: NCCL all-gather (tile flags, Q3), in-kernel peer-memory "
                                  f"reductions of the EM statistics over NVLink", "samples": N, "windows": int(res["n_windows"]),
                      "parallelism": f"sample-sharded x{world}", "calls_per_step": int(n_calls), "flagged_windows": int(res["n_flagged_windows"]),
                      "candidates": int(res["n_candidates"]), "parity_check": check},
           "clocks": clk, "gpu_launches": launches, "ms_device_per_step_rank0": float(np.mean(ms_dev))}
    emit_json(out)


# ----------------------------------------------------------------------------------------------------------------
# reference arm
# ----------------------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    if rank != 0:
        return
    binary = os.path.join(ROOT, "oracle", "_ref", "popdel_ref")
    cores = os.cpu_count() or 1
    N = args.samples
    slice_bp = int(min(args.ref_slice, args.length))          # >= 24 Mbp: several segments per process, start-up does not dominate
    cohort, _ = make_cohort(args.seed, N, slice_bp, args.dels_per_mbp, cores)      # (libpdsynth.so: nothing of the product is mapped here)
    tmp = tempfile.mkdtemp(prefix="popdel_ref_bench_")
    try:
        paths, lst = write_profiles(cohort, N, tmp, cores)
        kind = "reference" if os.path.exists(binary) else "port"

        def step():
            if kind == "reference":
                return run_reference_regions(binary, lst, tmp, slice_bp, cores)
            t0 = time.perf_counter()
            import oracle_api
            orc = oracle_api.load(os.path.join(ROOT, "oracle", "liboracle.so"))
            orc.call_files(paths, os.path.join(tmp, "dump.txt"))
            return time.perf_counter() - t0

        for _ in range(min(args.warmup, 1)):
            step()
        times = [step() for _ in range(args.steps)]
        dt = float(np.sum(times))
        evals = N * (slice_bp // 30)
        value = evals * args.steps / dt
        used = cores if kind == "reference" else 1
        out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
               "warmup": min(args.warmup, 1), "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "long double (x87)", "data": "synthetic",
               "config": workload_config(N, args.length, args.mixed, args.dels_per_mbp, world),
               "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": kind,
                                "sample": f"bounded sample of the workload: {N} samples x first {slice_bp} bp ({slice_bp // 30} windows per step), "
                                          f"gzip profile files on local disk -> VCF, {used} processes over contiguous -r regions"},
               "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit_json(out)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


_REAL_STDOUT = None


def emit_json(obj):
    """The ONE JSON line of the contract goes to the process's original stdout."""
    f = _REAL_STDOUT or sys.stdout
    f.write(json.dumps(obj) + "\n")
    f.flush()


def main():
    # Libraries chat on stdout (NCCL prints its version there at communicator creation): route fd 1 to stderr for the
    # whole run and keep the original stdout for the JSON line only.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--samples", type=int, default=100)
    ap.add_argument("--length", type=int, default=CHR21_LEN)
    ap.add_argument("--dels-per-mbp", type=float, default=2.0)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-slice", type=int, default=1_500_000)
    ap.add_argument("--ref-slice", type=int, default=24_000_000, help="bp of the workload the reference binary is timed on per step")
    ap.add_argument("--no-e2e-files", action="store_true")
    ap.add_argument("--output", default="unify", choices=["calls", "unify"], help="what the timed scan returns (see run_ours)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--shard-samples", action="store_true", help="sample-sharded cohort over the ranks (config 5 style) instead of window ranges")
    ap.add_argument("--check", action="store_true", help="--shard-samples: compare the merged calls with the CPU oracle (small cohorts)")
    ap.add_argument("--mixed", action="store_true", help="1-3 read groups per sample with mixed insert-size histograms")
    ap.add_argument("--device-gen", action="store_true", help="--shard-samples: generate the read pairs on the GPU (libpdsynth_cuda.so) and hand them "
                                                               "over with pd_contig_push_device (cohorts too large for the host generator)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (calls, per-sample rows, "
                                                          "significant windows) as DIR/<name>.npy in float64, at most 64 MB in all. "
                                                          "Window-range scan only: not with --impl reference (its output is VCF "
                                                          "text) or --shard-samples (each rank holds only its own samples' rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.shard_samples):
        ap.error("--dump-outputs covers the window-range scan (the default --impl ours without --shard-samples)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.shard_samples:
        run_sample_sharded(args, rank, world, local_rank)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
