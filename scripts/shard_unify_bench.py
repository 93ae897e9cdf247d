#!/usr/bin/env python
"""Sample-sharded cohort: window-call output versus merged variants (pd_set_unify on every rank), same contexts.

    torchrun --nproc_per_node 8 scripts/shard_unify_bench.py --samples 50000 --length 3000000 --device-gen
    torchrun --nproc_per_node 2 scripts/shard_unify_bench.py --samples 40 --length 1500000 --check

One rank per GPU (NCCL). The cohort is bench.py's (make_cohort / cohort_specs / plant, or the device generator with
--device-gen). After a warm-up of both modes the two outputs are timed twice each, alternating (calls, merged, calls,
merged): ms per step = wall time of --steps collective scans between barriers, max over ranks. Also per mode: the bytes
each rank's scan wrote to host memory (d2h_bytes), ms_unify (CUDA events around the merge stage incl. its exchanges),
the window-call and variant counts. --check (small cohorts): the oracle's unifyCalls on the gathered window calls ==
the merged variants. Prints one JSON line on rank 0 (and writes it to --out when given)."""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bench  # noqa: E402  (make_cohort, cohort_specs, plant, ClockSampler)


def card(local_rank):
    import torch
    name = torch.cuda.get_device_name(local_rank)
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = None
    return dict(name=name, power_limit_and_max_sm_clock=out)


def main():
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)                               # NCCL prints on stdout; the JSON line goes to the original one
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=50000)
    ap.add_argument("--length", type=int, default=3_000_000)
    ap.add_argument("--dels-per-mbp", type=float, default=2.0)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--cover", type=float, default=0.5, help="-c: min_relative_window_cover of the merge")
    ap.add_argument("--device-gen", action="store_true", help="generate the read pairs on the GPU (libpdsynth_cuda.so)")
    ap.add_argument("--check", action="store_true", help="compare the merged variants with the oracle's unifyCalls (small cohorts)")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch
    import torch.distributed as dist
    from popdel_b200 import api
    rank, world, local_rank = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    assert world >= 2, "run under torchrun with >= 2 ranks (one per GPU)"
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    threads = max(1, (os.cpu_count() or 8) // world)
    N, L = args.samples, args.length
    spr = api.split_samples(N, world)
    s0 = sum(spr[:rank])
    # the same set-up as bench.py --shard-samples
    hdr_len = min(L, 300_000) if args.device_gen else L
    cohort, dels = bench.make_cohort(args.seed, N, L, args.dels_per_mbp, threads, sample_range=(s0, s0 + spr[rank]), gen_length=hdr_len)
    params = api.CallParameters()
    specs = bench.cohort_specs(args.seed, N)
    every = [api.ReadGroup(sample=sp[0], median=int(sp[2]), read_length=150, stddev=sp[3], offset=0, values=np.zeros(3), min_prob=0.0,
                           lower_quantile_dist=0, upper_quantile_dist=0) for sp in specs]
    params.finalize(every)
    min_init = np.array([r.min_init_del_len for r in every], dtype=np.uint32)
    mean_sd = float(np.mean([r.stddev for r in every]))            # meanStddev over every read group of the cohort
    rgs = api.read_groups_from_headers([[c[3] for c in cohort if c[4] == s] for s in range(s0, s0 + spr[rank])],
                                       api.CallParameters(min_len=params.min_len))
    uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        uid.copy_(torch.frombuffer(bytearray(api.shard_unique_id()), dtype=torch.uint8))
    dist.broadcast(uid, 0)
    sc = api.Scanner(params, rgs, spr[rank], device=local_rank)
    sc.attach_nccl(rank, world, spr, min_init, bytes(uid.cpu().numpy()))
    sc.begin_contig(0)
    sc.reserve_windows(L // 30 + 2)
    gen = None
    if args.device_gen:
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

    def set_mode(mode):
        if mode == "merged":
            sc.set_unify(mean_stddev=mean_sd, min_relative_window_cover=args.cover, output_failed=False)
        else:
            sc.set_unify(None)

    check = None
    if args.check:
        got = {}
        for mode in ("calls", "merged"):
            set_mode(mode)
            r = sc.scan(copy=True)
            parts = [None] * world
            dist.all_gather_object(parts, dict(calls=r["calls"], per_sample=r["per_sample"], sig=r["significant_windows"]))
            got[mode] = parts
        if rank == 0:
            import oracle_api
            from parity import assert_calls_equal
            orc = oracle_api.load(os.path.join(ROOT, "oracle", "liboracle.so"))
            raw, uni = got["calls"], got["merged"]
            for p in raw[1:]:
                assert np.array_equal(p["calls"], raw[0]["calls"]), "ranks disagree on the window calls"
            for p in uni[1:]:
                assert p["calls"].tobytes() == uni[0]["calls"].tobytes() and np.array_equal(p["sig"], uni[0]["sig"]), "ranks disagree on the variants"
            ref_calls, ref_ps, ref_sig = orc.unify_segments(raw[0]["calls"], np.concatenate([p["per_sample"] for p in raw], axis=1),
                                                           mean_sd, args.cover, False)
            assert_calls_equal(uni[0]["calls"], np.concatenate([p["per_sample"] for p in uni], axis=1), ref_calls, ref_ps)
            assert np.array_equal(uni[0]["sig"], ref_sig)
            check = (f"merged variants of {world} ranks == oracle unifyCalls of the gathered window calls ({len(raw[0]['calls'])} window calls "
                     f"-> {len(ref_calls)} variants, integers bit-exact, LR/AF 1e-6)")

    for mode in ("calls", "merged"):
        set_mode(mode)
        for _ in range(args.warmup):
            sc.scan(copy=False)
    clocks = bench.ClockSampler(local_rank if rank == 0 else None)
    clocks.start()
    runs = []
    for rep in range(2):
        for mode in ("calls", "merged"):
            set_mode(mode)
            dist.barrier(); torch.cuda.synchronize()
            t0 = time.perf_counter()
            ms_unify = []
            for _ in range(args.steps):
                r = sc.scan(copy=False)
                ms_unify.append(r["ms_unify"])
            dist.barrier(); torch.cuda.synchronize()
            dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            mine = dict(d2h_bytes=int(r["d2h_bytes"]), ms_unify=float(np.mean(ms_unify)), n_calls=int(len(r["calls"])),
                        n_window_calls=int(r["n_window_calls"]), ms_device=float(r["ms_total"]))
            every_rank = [None] * world
            dist.all_gather_object(every_rank, mine)
            runs.append(dict(mode=mode, rep=rep, ms_per_step=float(dt.item()) / args.steps * 1e3,
                             d2h_bytes_per_rank=[e["d2h_bytes"] for e in every_rank],
                             ms_unify_rank0=every_rank[0]["ms_unify"], ms_unify_max=max(e["ms_unify"] for e in every_rank),
                             n_calls=every_rank[0]["n_calls"], n_window_calls=every_rank[0]["n_window_calls"],
                             ms_device_per_step_rank0=every_rank[0]["ms_device"]))
    clk = clocks.stop()
    info = card(local_rank)
    n_windows = int(r["n_windows"])
    sc.close()
    if gen is not None:
        gen.close()
    dist.barrier()
    dist.destroy_process_group()
    if rank != 0:
        return
    best = {m: min(x["ms_per_step"] for x in runs if x["mode"] == m) for m in ("calls", "merged")}
    out = {"what": "sample-sharded scan: window calls vs merged variants (pd_set_unify), same contexts, alternating",
           "samples": N, "length_bp": L, "windows": n_windows, "gpus": world, "samples_per_gpu": spr[0], "steps": args.steps,
           "warmup": args.warmup, "device_gen": args.device_gen, "cover": args.cover, "card": info, "clocks": clk,
           "runs": runs, "ms_per_step_best": best, "parity_check": check}
    line = json.dumps(out)
    real_stdout.write(line + "\n")
    real_stdout.flush()
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
