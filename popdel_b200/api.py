"""Python binding of the scan library (include/popdel_b200.h) and the host-side mirror of the reference's
parameter handling for `popdel call`.

Everything that computes on read pairs goes through the C ABI of `libpopdel_b200.so` (hand-written CUDA, sm_100a).
There is no CPU scan path: creating a `Scanner` on a box without a usable CUDA device raises `ScanError`
(only `device=-1` host-only contexts, used to validate the packed layout, work without a GPU).
"""
from __future__ import annotations

import ctypes as C
import math
import os
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("POPDEL_B200_LIB") or os.path.join(_HERE, "libpopdel_b200.so")      # (override: A/B runs of two builds)


class ScanError(RuntimeError):
    pass


class PdParams(C.Structure):
    _fields_ = [("iterations", C.c_uint32), ("min_len", C.c_uint32), ("min_lr", C.c_double),
                ("min_sample_fraction", C.c_double), ("window_size", C.c_uint32), ("window_buffer", C.c_uint32),
                ("somatic", C.c_int32), ("window_wise", C.c_int32)]


class PdRg(C.Structure):
    _fields_ = [("sample", C.c_uint32), ("median", C.c_uint32), ("read_length", C.c_uint32), ("stddev", C.c_double),
                ("offset", C.c_int32), ("len", C.c_uint32), ("values", C.POINTER(C.c_double)), ("min_prob", C.c_double),
                ("lower_quantile_dist", C.c_uint32), ("upper_quantile_dist", C.c_uint32), ("max_load", C.c_uint32),
                ("min_init_del_len", C.c_uint32)]


class PdResult(C.Structure):
    _fields_ = [("n_calls", C.c_uint64), ("calls", C.c_void_p), ("per_sample", C.POINTER(C.c_uint32)),
                ("n_windows", C.c_uint64), ("n_flagged_windows", C.c_uint64), ("n_candidates", C.c_uint64),
                ("n_reads", C.c_uint64), ("algorithmic_bytes", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("n_kernel_launches", C.c_uint64),
                ("ms_h2d", C.c_float), ("ms_screen", C.c_float), ("ms_genotype", C.c_float), ("ms_d2h", C.c_float),
                ("ms_total", C.c_float), ("ms_stream", C.c_float),
                ("significant_windows", C.POINTER(C.c_uint32)), ("n_window_calls", C.c_uint64), ("ms_unify", C.c_float),
                ("ms_em", C.c_float), ("n_em_pairs_timed", C.c_uint32), ("n_screened_windows", C.c_uint64),
                ("n_known_pairs", C.c_uint64)]


class PdUnifyParams(C.Structure):
    _fields_ = [("mean_stddev", C.c_double), ("min_relative_window_cover", C.c_double), ("output_failed", C.c_int32),
                ("reserved", C.c_int32)]


CALL_DTYPE = np.dtype([("initial_length", "<u4"), ("iterations", "<u4"), ("deletion_length", "<u4"), ("filter", "<u4"),
                       ("lr", "<f8"), ("frequency", "<f8"), ("window_position", "<u4"), ("position", "<u4"),
                       ("end_position", "<u4"), ("segment", "<u4")])

EXPORTS = ["pd_process_histogram", "pd_create", "pd_create_error", "pd_destroy", "pd_last_error", "pd_contig_begin",
           "pd_contig_push", "pd_contig_push_pinned", "pd_contig_push_compact", "pd_contig_push_compact32", "pd_contig_push_device", "pd_contig_upload", "pd_contig_scan", "pd_contig_window_count",
           "pd_debug_host_window_sums", "pd_debug_cap_replay", "pd_contig_reserve_windows", "pd_shard_unique_id", "pd_shard_attach_nccl",
           "pd_shard_attach_group", "pd_shard_group_scan", "pd_set_unify", "pd_device_warmup", "pd_set_staging"]

_lib = None


class PdShardInfo(C.Structure):
    _fields_ = [("rank", C.c_uint32), ("world", C.c_uint32), ("n_samples_global", C.c_uint32), ("n_rg_global", C.c_uint32),
                ("min_init_global", C.POINTER(C.c_uint32)), ("samples_per_rank", C.POINTER(C.c_uint32))]


def load_library(path: str = LIB_PATH):
    """Loads libpopdel_b200.so; raises ScanError when it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(path):
        raise ScanError(f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(nvcc, sm_100a). popdel_b200 has no CPU implementation of the scan.")
    lib = C.CDLL(path)
    lib.pd_process_histogram.restype = C.c_double
    lib.pd_process_histogram.argtypes = [C.POINTER(C.c_double), C.c_uint32, C.c_int32, C.c_uint32, C.c_uint32, C.c_int,
                                         C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    lib.pd_create.restype = C.c_void_p
    lib.pd_create.argtypes = [C.POINTER(PdParams), C.c_uint32, C.c_uint32, C.POINTER(PdRg), C.c_int]
    lib.pd_create_error.restype = C.c_char_p
    lib.pd_destroy.argtypes = [C.c_void_p]
    lib.pd_last_error.restype = C.c_char_p
    lib.pd_last_error.argtypes = [C.c_void_p]
    lib.pd_contig_begin.argtypes = [C.c_void_p, C.c_uint32]
    lib.pd_contig_push.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.POINTER(C.c_uint32), C.POINTER(C.c_int32)]
    lib.pd_contig_push_pinned.argtypes = lib.pd_contig_push.argtypes
    lib.pd_contig_push_compact32.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.POINTER(C.c_uint32), C.c_uint32, C.POINTER(C.c_uint32)]
    lib.pd_contig_push_device.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p]
    lib.pd_contig_push_compact.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.POINTER(C.c_uint16), C.POINTER(C.c_uint8),
                                           C.c_uint32, C.POINTER(C.c_uint32)]
    lib.pd_contig_upload.argtypes = [C.c_void_p]
    lib.pd_contig_scan.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(PdResult)]
    lib.pd_contig_window_count.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
    lib.pd_debug_host_window_sums.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64, C.POINTER(C.c_int64)]
    lib.pd_contig_reserve_windows.argtypes = [C.c_void_p, C.c_uint64]
    lib.pd_shard_unique_id.argtypes = [C.POINTER(C.c_uint8)]
    lib.pd_shard_attach_nccl.argtypes = [C.c_void_p, C.POINTER(PdShardInfo), C.POINTER(C.c_uint8)]
    lib.pd_shard_attach_group.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.POINTER(PdShardInfo)]
    lib.pd_shard_group_scan.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.c_uint64, C.c_uint64, C.POINTER(PdResult)]
    lib.pd_set_unify.argtypes = [C.c_void_p, C.POINTER(PdUnifyParams)]
    lib.pd_set_staging.argtypes = [C.c_void_p, C.c_int]
    lib.pd_device_warmup.argtypes = [C.c_int]
    _lib = lib
    return lib


_synth = None


def load_synth_library():
    global _synth
    if _synth is None:
        path = os.path.join(_HERE, "libpdsynth.so")
        if not os.path.exists(path):
            raise ScanError(f"{path} is missing: build it with `make -C popdel_b200/csrc`")
        _synth = C.CDLL(path)
        _synth.pd_synth_read_group.restype = C.c_int64
        _synth.pd_synth_read_group.argtypes = [C.c_uint64, C.c_uint32, C.c_double, C.c_double, C.c_uint32, C.c_double,
                                               C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32),
                                               C.POINTER(C.c_uint32), C.POINTER(C.c_uint8), C.POINTER(C.c_uint32),
                                               C.POINTER(C.c_int32), C.c_uint64]
    return _synth


def process_histogram(counts, offset: int, median: int, read_length: int, smoothing: bool = True,
                      pseudo_count_fraction: int = 500):
    """processHistogram(hist, 256, smoothing, f) of the reference (insert_histogram_popdel.h:974-986).
    Returns (values, min_prob, lower_quantile_dist, upper_quantile_dist)."""
    lib = load_library()
    v = np.ascontiguousarray(counts, dtype=np.float64).copy()
    lq, uq = C.c_uint32(0), C.c_uint32(0)
    mp = lib.pd_process_histogram(v.ctypes.data_as(C.POINTER(C.c_double)), v.size, int(offset), int(median),
                                  int(read_length), int(smoothing), int(pseudo_count_fraction), C.byref(lq), C.byref(uq))
    return v, mp, lq.value, uq.value


@dataclass
class ReadGroup:
    """One read group of the cohort = one Histogram of the reference plus its per-RG call parameters."""
    sample: int
    median: int
    read_length: int
    stddev: float
    offset: int
    values: np.ndarray            # processed histogram
    min_prob: float
    lower_quantile_dist: int
    upper_quantile_dist: int
    max_load: int = 100
    min_init_del_len: int = 0
    name: str = ""

    def as_dict(self):
        return dict(sample=self.sample, median=self.median, read_length=self.read_length, stddev=self.stddev,
                    offset=self.offset, values=self.values, min_prob=self.min_prob,
                    lower_quantile_dist=self.lower_quantile_dist, upper_quantile_dist=self.upper_quantile_dist,
                    max_load=self.max_load, min_init_del_len=self.min_init_del_len)


@dataclass
class CallParameters:
    """Defaults and derived values of PopDelCallParameters (popdel_call/parameter_parsing_popdel_call.h:184-209,
    popdel_call/parameter_calculation_popdel_call.h:16-81,160-204)."""
    iterations: int = 15
    prior: float = 0.0001
    min_len: Optional[int] = None              # -m; default 95th percentile of the initial lengths
    min_init_len: Optional[int] = None         # -l; default round(4 * stddev) per read group
    min_sample_fraction: float = 0.1
    window_size: int = 30
    window_buffer: int = 200000
    somatic: bool = False
    window_wise: bool = False
    default_max_load: int = 100                # -a; 0 disables the cap
    smoothing: bool = True
    pseudo_count_fraction: int = 500
    min_lr: float = field(init=False, default=0.0)

    def finalize(self, rgs: List[ReadGroup]) -> None:
        """loadAndCalculateParameters: min init lengths, min length, LR threshold, max load."""
        for r in rgs:
            r.min_init_del_len = int(self.min_init_len) if self.min_init_len is not None else int(math.floor(4 * r.stddev + 0.5))
            r.max_load = 0xFFFFFFFF if self.default_max_load == 0 else int(self.default_max_load)
        if self.min_len is None:
            v = sorted(r.min_init_del_len for r in rgs)
            n = len(v)
            j = int(math.floor(n * 0.95))
            self.min_len = int(math.floor(1.0 * (v[j] if j != n * 0.95 else v[j - 1]) + 0.5))
        self.min_lr = (6.6349 / 2.0) - math.log(self.prior / (1 - self.prior))

    def as_dict(self):
        return dict(iterations=self.iterations, min_len=int(self.min_len), min_lr=self.min_lr,
                    min_sample_fraction=self.min_sample_fraction, window_size=self.window_size,
                    window_buffer=self.window_buffer, somatic=int(self.somatic), window_wise=int(self.window_wise))


def read_groups_from_headers(headers: Sequence[Sequence[dict]], params: CallParameters) -> List[ReadGroup]:
    """headers[s] = read-group header dicts of sample s (profile_format.rg_meta_from / read_profile):
    processes every histogram like loadInsertSizeHistograms (insert_histogram_popdel.h:992-1095)."""
    out: List[ReadGroup] = []
    for s, metas in enumerate(headers):
        for m in metas:
            vals, mp, lq, uq = process_histogram(m["hist_counts"], m["hist_start"], m["median"], m["read_length"],
                                                 params.smoothing, params.pseudo_count_fraction)
            out.append(ReadGroup(sample=s, median=int(m["median"]), read_length=int(m["read_length"]),
                                 stddev=float(m["stddev"]), offset=int(m["hist_start"]), values=vals, min_prob=mp,
                                 lower_quantile_dist=lq, upper_quantile_dist=uq, name=m.get("name", "")))
    params.finalize(out)
    return out


class Scanner:
    """One scan context (pd_ctx) on one GPU."""

    def __init__(self, params: CallParameters, rgs: List[ReadGroup], n_samples: int, device: int = 0):
        self.lib = load_library()
        self.n_samples, self.n_rg = int(n_samples), len(rgs)
        self._keep = [np.ascontiguousarray(r.values, dtype=np.float64) for r in rgs]
        arr = (PdRg * len(rgs))()
        for i, r in enumerate(rgs):
            arr[i] = PdRg(r.sample, r.median, r.read_length, r.stddev, r.offset, self._keep[i].size,
                          self._keep[i].ctypes.data_as(C.POINTER(C.c_double)), r.min_prob, r.lower_quantile_dist,
                          r.upper_quantile_dist, r.max_load, r.min_init_del_len)
        p = PdParams(**params.as_dict())
        self.ctx = self.lib.pd_create(C.byref(p), self.n_samples, self.n_rg, arr, int(device))
        if not self.ctx:
            raise ScanError(self.lib.pd_create_error().decode())

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.pd_destroy(self.ctx)
            self.ctx = None

    __del__ = close

    def _check(self, rc):
        if rc != 0:
            raise ScanError(f"[{rc}] {self.lib.pd_last_error(self.ctx).decode()}")

    def begin_contig(self, anchor: int):
        self._check(self.lib.pd_contig_begin(self.ctx, int(anchor)))

    def push(self, rg: int, pos: np.ndarray, dev: np.ndarray):
        pos = np.ascontiguousarray(pos, dtype=np.uint32)
        dev = np.ascontiguousarray(dev, dtype=np.int32)
        assert pos.size == dev.size
        self._check(self.lib.pd_contig_push(self.ctx, int(rg), pos.size, pos.ctypes.data_as(C.POINTER(C.c_uint32)),
                                            dev.ctypes.data_as(C.POINTER(C.c_int32))))

    def push_pinned(self, rg: int, pos: np.ndarray, dev: np.ndarray):
        """pd_contig_push_pinned: `pos` (uint32) / `dev` (int32) must be C-contiguous views of page-locked memory and
        stay alive and unchanged until upload()/scan() returns."""
        assert pos.dtype == np.uint32 and dev.dtype == np.int32 and pos.flags.c_contiguous and dev.flags.c_contiguous
        assert pos.size == dev.size
        self._pinned_keep = getattr(self, "_pinned_keep", {})
        self._pinned_keep[rg] = (pos, dev)
        self._check(self.lib.pd_contig_push_pinned(self.ctx, int(rg), pos.size, pos.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                   dev.ctypes.data_as(C.POINTER(C.c_int32))))

    def push_compact(self, rg: int, pos_lo: np.ndarray, dev24: np.ndarray, blk_first: np.ndarray):
        """pd_contig_push_compact (5 bytes per read pair over PCIe, see compact_encode): C-contiguous views of page-locked
        memory that stay alive and unchanged until upload()/scan() returns."""
        assert pos_lo.dtype == np.uint16 and dev24.dtype == np.uint8 and blk_first.dtype == np.uint32
        assert pos_lo.flags.c_contiguous and dev24.flags.c_contiguous and blk_first.flags.c_contiguous
        assert dev24.size == 3 * pos_lo.size and blk_first.size >= 2
        self._pinned_keep = getattr(self, "_pinned_keep", {})
        self._pinned_keep[rg] = (pos_lo, dev24, blk_first)
        self._check(self.lib.pd_contig_push_compact(self.ctx, int(rg), pos_lo.size, pos_lo.ctypes.data_as(C.POINTER(C.c_uint16)),
                                                    dev24.ctypes.data_as(C.POINTER(C.c_uint8)), blk_first.size - 1,
                                                    blk_first.ctypes.data_as(C.POINTER(C.c_uint32))))

    def push_compact32(self, rg: int, words: np.ndarray, blk_first: np.ndarray):
        """pd_contig_push_compact32 (4 bytes per read pair over PCIe, see compact32_encode): C-contiguous views of page-locked
        memory that stay alive and unchanged until upload()/scan() returns."""
        assert words.dtype == np.uint32 and blk_first.dtype == np.uint32 and words.flags.c_contiguous and blk_first.flags.c_contiguous
        assert blk_first.size >= 2
        self._pinned_keep = getattr(self, "_pinned_keep", {})
        self._pinned_keep[rg] = (words, blk_first)
        self._check(self.lib.pd_contig_push_compact32(self.ctx, int(rg), words.size, words.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                      blk_first.size - 1, blk_first.ctypes.data_as(C.POINTER(C.c_uint32))))

    def push_device(self, rg: int, n: int, d_pos: int, d_dev: int):
        """pd_contig_push_device: d_pos (uint32[n]) / d_dev (int32[n]) are DEVICE addresses on this scanner's GPU (e.g.
        torch_tensor.data_ptr()) that stay valid and unchanged until upload()/scan() returns."""
        self._check(self.lib.pd_contig_push_device(self.ctx, int(rg), int(n), C.c_void_p(int(d_pos) if n else 0), C.c_void_p(int(d_dev) if n else 0)))

    def upload(self):
        self._check(self.lib.pd_contig_upload(self.ctx))

    def window_count(self) -> int:
        n = C.c_uint64(0)
        self._check(self.lib.pd_contig_window_count(self.ctx, C.byref(n)))
        return n.value

    def scan(self, first_window: int = 0, n_windows: int = 0, copy: bool = True) -> dict:
        """Runs the scan. With copy=False `calls` / `per_sample` are views of library-owned (pinned) memory that stay
        valid until the next call on this scanner."""
        res = PdResult()
        self._check(self.lib.pd_contig_scan(self.ctx, int(first_window), int(n_windows), C.byref(res)))
        n = res.n_calls
        if n and not copy:
            calls = np.frombuffer((C.c_char * (n * CALL_DTYPE.itemsize)).from_address(res.calls), dtype=CALL_DTYPE)
            per = np.ctypeslib.as_array(res.per_sample, shape=(n, self.n_samples, 13))
        else:
            calls = np.zeros(n, dtype=CALL_DTYPE)
            per = np.zeros((n, self.n_samples, 13), dtype=np.uint32)
            if n:
                C.memmove(calls.ctypes.data, res.calls, n * CALL_DTYPE.itemsize)
                C.memmove(per.ctypes.data, res.per_sample, per.nbytes)
        sig = None
        if res.significant_windows:
            sig = np.ctypeslib.as_array(res.significant_windows, shape=(max(n, 1),))[:n].copy()
        return dict(calls=calls, per_sample=per, n_windows=res.n_windows, n_flagged_windows=res.n_flagged_windows,
                    n_candidates=res.n_candidates, n_reads=res.n_reads, algorithmic_bytes=res.algorithmic_bytes,
                    h2d_bytes=res.h2d_bytes, d2h_bytes=res.d2h_bytes, n_kernel_launches=res.n_kernel_launches,
                    ms_h2d=res.ms_h2d, ms_screen=res.ms_screen, ms_genotype=res.ms_genotype, ms_total=res.ms_total,
                    ms_stream=res.ms_stream, significant_windows=sig, n_window_calls=res.n_window_calls, ms_unify=res.ms_unify,
                    ms_em=res.ms_em, n_em_pairs_timed=res.n_em_pairs_timed, n_screened_windows=res.n_screened_windows,
                    n_known_pairs=res.n_known_pairs)

    def set_unify(self, mean_stddev=None, min_relative_window_cover: float = 0.5, output_failed: bool = False):
        """pd_set_unify: scans return the merged variants of every segment (unifyCalls, utils_popdel.h:567-654, run on the
        device); mean_stddev=None switches back to window calls. On a sample-sharded scanner (attach_nccl, ShardGroup)
        every rank must use the same settings: each rank then returns the cohort's variants with its own samples' rows."""
        if mean_stddev is None:
            self._check(self.lib.pd_set_unify(self.ctx, None))
            return
        p = PdUnifyParams(float(mean_stddev), float(min_relative_window_cover), int(bool(output_failed)), 0)
        self._check(self.lib.pd_set_unify(self.ctx, C.byref(p)))

    def set_staging(self, pinned: bool):
        """pd_set_staging: page-locked (default) or pageable staging buffers for push()."""
        self._check(self.lib.pd_set_staging(self.ctx, int(bool(pinned))))

    def reserve_windows(self, n_windows: int):
        self._check(self.lib.pd_contig_reserve_windows(self.ctx, int(n_windows)))

    def _result_dict(self, res, copy=True) -> dict:
        n = res.n_calls
        calls = np.zeros(n, dtype=CALL_DTYPE)
        per = np.zeros((n, self.n_samples, 13), dtype=np.uint32)
        if n:
            C.memmove(calls.ctypes.data, res.calls, n * CALL_DTYPE.itemsize)
            C.memmove(per.ctypes.data, res.per_sample, per.nbytes)
        sig = None
        if res.significant_windows:
            sig = np.ctypeslib.as_array(res.significant_windows, shape=(max(n, 1),))[:n].copy()
        return dict(calls=calls, per_sample=per, n_windows=res.n_windows, n_flagged_windows=res.n_flagged_windows,
                    n_candidates=res.n_candidates, n_reads=res.n_reads, algorithmic_bytes=res.algorithmic_bytes,
                    h2d_bytes=res.h2d_bytes, d2h_bytes=res.d2h_bytes, n_kernel_launches=res.n_kernel_launches,
                    ms_h2d=res.ms_h2d, ms_screen=res.ms_screen, ms_genotype=res.ms_genotype, ms_total=res.ms_total,
                    ms_stream=res.ms_stream, significant_windows=sig, n_window_calls=res.n_window_calls, ms_unify=res.ms_unify,
                    ms_em=res.ms_em, n_em_pairs_timed=res.n_em_pairs_timed, n_screened_windows=res.n_screened_windows,
                    n_known_pairs=res.n_known_pairs)

    def attach_nccl(self, rank: int, world: int, samples_per_rank, min_init_global, unique_id: bytes):
        """Sample sharding, one process per GPU (pd_shard_attach_nccl; collective)."""
        self._shard_keep = (np.ascontiguousarray(min_init_global, dtype=np.uint32), np.ascontiguousarray(samples_per_rank, dtype=np.uint32),
                            (C.c_uint8 * 128).from_buffer_copy(bytes(unique_id)))
        mi, spr, uid = self._shard_keep
        info = PdShardInfo(int(rank), int(world), int(spr.sum()), mi.size, mi.ctypes.data_as(C.POINTER(C.c_uint32)),
                           spr.ctypes.data_as(C.POINTER(C.c_uint32)))
        self._check(self.lib.pd_shard_attach_nccl(self.ctx, C.byref(info), uid))

    def debug_host_window_sums(self, rg: int, first_window: int, n_windows: int) -> np.ndarray:
        out = np.zeros((int(n_windows), 3), dtype=np.int64)
        self._check(self.lib.pd_debug_host_window_sums(self.ctx, int(rg), int(first_window), int(n_windows),
                                                       out.ctypes.data_as(C.POINTER(C.c_int64))))
        return out


def synth_read_group(seed: int, rg_index: int, mu: float, sigma: float, read_length: int, pairs_per_bp: float,
                     first_pos: int, end_pos: int, del_start=(), del_len=(), del_genotype=()):
    """pd_synth_read_group (libpdsynth.so, include/pdsynth.h: test / benchmark infrastructure, not the scan library):
    returns (pos uint32, isize int32), sorted by (pos, isize). Releases the GIL."""
    lib = load_synth_library()
    ds = np.ascontiguousarray(del_start, dtype=np.uint32)
    dl = np.ascontiguousarray(del_len, dtype=np.uint32)
    dg = np.ascontiguousarray(del_genotype, dtype=np.uint8)
    span = int(end_pos) - int(first_pos)
    cap = int(span * pairs_per_bp * 1.05) + 100000
    pos = np.empty(cap, dtype=np.uint32)
    isz = np.empty(cap, dtype=np.int32)
    n = lib.pd_synth_read_group(int(seed), int(rg_index), float(mu), float(sigma), int(read_length), float(pairs_per_bp),
                                int(first_pos), int(end_pos), ds.size, ds.ctypes.data_as(C.POINTER(C.c_uint32)),
                                dl.ctypes.data_as(C.POINTER(C.c_uint32)), dg.ctypes.data_as(C.POINTER(C.c_uint8)),
                                pos.ctypes.data_as(C.POINTER(C.c_uint32)), isz.ctypes.data_as(C.POINTER(C.c_int32)), cap)
    if n < 0:
        raise ScanError(f"pd_synth_read_group failed ({n})")
    return pos[:n], isz[:n]


class PdSynthRg(C.Structure):
    _fields_ = [("mu", C.c_double), ("sigma", C.c_double), ("pairs_per_bp", C.c_double), ("rg_index", C.c_uint32), ("sample", C.c_uint32),
                ("read_length", C.c_uint32), ("median", C.c_uint32)]


class SynthDevice:
    """pdsynth_dev_* (libpdsynth_cuda.so, include/pdsynth.h): the counter-based generator on the GPU. generate() returns
    (total, d_pos, d_dev, rg_start): device addresses of uint32 positions / int32 deviations owned by this object (valid until
    the next generate()) and the host array of read-group offsets -- what Scanner.push_device takes."""

    def __init__(self, device: int = 0):
        path = os.path.join(_HERE, "libpdsynth_cuda.so")
        if not os.path.exists(path):
            raise ScanError(f"{path} not built (make -C popdel_b200/csrc)")
        self.lib = C.CDLL(path)
        self.lib.pdsynth_dev_create.restype = C.c_void_p
        self.lib.pdsynth_dev_create.argtypes = [C.c_int]
        self.lib.pdsynth_dev_destroy.argtypes = [C.c_void_p]
        self.lib.pdsynth_dev_generate.restype = C.c_int64
        self.lib.pdsynth_dev_generate.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.POINTER(PdSynthRg), C.c_uint32, C.c_uint32, C.c_uint32,
                                                  C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint8), C.c_uint32,
                                                  C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
        self.h = self.lib.pdsynth_dev_create(int(device))
        if not self.h:
            raise ScanError("pdsynth_dev_create failed (no usable CUDA device)")

    def close(self):
        if self.h:
            self.lib.pdsynth_dev_destroy(self.h)
            self.h = None

    def to_host(self, d_ptr: int, n: int, dtype) -> np.ndarray:
        out = np.empty(n, dtype=dtype)
        self.lib.pdsynth_dev_copy_to_host.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
        if self.lib.pdsynth_dev_copy_to_host(self.h, out.ctypes.data_as(C.c_void_p), C.c_void_p(d_ptr), out.nbytes) != 0:
            raise ScanError("pdsynth_dev_copy_to_host failed")
        return out

    def generate(self, seed, specs, first_pos, end_pos, del_start=(), del_len=(), del_genotype=None, n_samples=1):
        """specs: sequence of (sample, rg_index, mu, sigma, pairs_per_bp[, read_length]); del_genotype: uint8 [n_dels, n_samples]."""
        arr = (PdSynthRg * len(specs))()
        for i, sp in enumerate(specs):
            s, g, mu, sd, dens = sp[:5]
            arr[i] = PdSynthRg(float(mu), float(sd), float(dens), int(g), int(s), int(sp[5]) if len(sp) > 5 else 150, int(mu))
        ds = np.ascontiguousarray(del_start, dtype=np.uint32)
        dl = np.ascontiguousarray(del_len, dtype=np.uint32)
        gt = np.ascontiguousarray(del_genotype if del_genotype is not None else np.zeros((ds.size, n_samples)), dtype=np.uint8)
        assert gt.shape == (ds.size, n_samples) or ds.size == 0
        rg_start = np.zeros(len(specs) + 1, dtype=np.uint64)
        dp, dd = C.c_void_p(0), C.c_void_p(0)
        n = self.lib.pdsynth_dev_generate(self.h, int(seed), len(specs), arr, int(first_pos), int(end_pos), ds.size,
                                          ds.ctypes.data_as(C.POINTER(C.c_uint32)), dl.ctypes.data_as(C.POINTER(C.c_uint32)),
                                          gt.ctypes.data_as(C.POINTER(C.c_uint8)), int(n_samples), C.byref(dp), C.byref(dd),
                                          rg_start.ctypes.data_as(C.POINTER(C.c_uint64)))
        if n < 0:
            raise ScanError(f"pdsynth_dev_generate failed ({n})")
        return int(n), int(dp.value or 0), int(dd.value or 0), rg_start


def compact_encode(pos: np.ndarray, dev: np.ndarray):
    """(pos uint32 sorted, dev int32) -> (pos_lo uint16, dev24 uint8[3n], blk_first uint32) of pd_contig_push_compact: what a
    profile decoder can emit directly (the file stores a u8 offset per 256-bp window and an i32 deviation)."""
    pos = np.ascontiguousarray(pos, dtype=np.uint32)
    dev = np.ascontiguousarray(dev, dtype=np.int32)
    assert dev.size == 0 or (int(dev.min()) >= -(1 << 23) and int(dev.max()) < (1 << 23))
    nblk = (int(pos[-1]) >> 16) + 1 if pos.size else 1
    blk_first = np.searchsorted(pos >> 16, np.arange(nblk + 1, dtype=np.uint32), side="left").astype(np.uint32)
    pos_lo = (pos & 0xFFFF).astype(np.uint16)
    dev24 = np.ascontiguousarray(dev.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :3]).reshape(-1)
    return pos_lo, dev24, blk_first


def compact32_encode(pos: np.ndarray, dev: np.ndarray):
    """(pos uint32 sorted, dev int32 with |dev| < 2^23) -> (words uint32, blk_first uint32) of pd_contig_push_compact32:
    word = dev << 8 | pos & 0xFF, blk_first[b] = first read pair of 256-bp block b -- the profile file's own granularity."""
    pos = np.ascontiguousarray(pos, dtype=np.uint32)
    dev = np.ascontiguousarray(dev, dtype=np.int32)
    assert dev.size == 0 or (int(dev.min()) >= -(1 << 23) and int(dev.max()) < (1 << 23))
    words = ((dev.astype(np.uint32) << np.uint32(8)) | (pos & np.uint32(0xFF))).astype(np.uint32)
    nb = int(pos[-1] >> 8) + 1 if pos.size else 1
    blk = np.searchsorted(pos >> np.uint32(8), np.arange(nb + 1, dtype=np.uint32), side="left").astype(np.uint32)
    return words, blk


def _page_locked(a: np.ndarray) -> np.ndarray:
    """A page-locked copy of `a` (torch pin_memory; the push_pinned / push_compact contract). Falls back to the array itself
    when torch has no CUDA runtime (the copies are then staged by the driver: slower, same result)."""
    try:
        import torch
        kinds = {np.dtype(np.uint32): np.int32, np.dtype(np.uint16): np.int16}
        view = a.view(kinds.get(a.dtype, a.dtype))
        t = torch.from_numpy(np.ascontiguousarray(view)).pin_memory()
        out = t.numpy().view(a.dtype)
        _page_locked.keep.append(t)
        if len(_page_locked.keep) > 4096:
            del _page_locked.keep[:2048]
        return out
    except Exception:
        return a


_page_locked.keep = []


def cohort_anchor(samples) -> int:
    """First 30-bp window over all samples (getFirstWindowCoordinate, load_profile_popdel_call.h:291-350)."""
    first = [int(rg.pos[0]) for s in samples for rg in s.read_groups if rg.pos.size]
    return (min(first) // 30) * 30


def scan_cohort(samples, params: CallParameters, device: int = 0, first_window: int = 0, n_windows: int = 0,
                pinned: bool = False, unify: dict = None):
    """Convenience: whole in-memory cohort (popdel_b200.simulate objects) -> window calls of one contig, or -- with
    unify=dict(mean_stddev=..., min_relative_window_cover=..., output_failed=...) -- the merged variants."""
    rgs = read_groups_from_headers([[dict(name=rg.spec.name, median=rg.median, stddev=rg.stddev,
                                          read_length=rg.spec.read_length, hist_start=rg.hist_start,
                                          hist_end=rg.hist_end, hist_counts=rg.hist_counts) for rg in s.read_groups]
                                    for s in samples], params)
    sc = Scanner(params, rgs, len(samples), device)
    try:
        if unify:
            sc.set_unify(**unify)
        sc.begin_contig(cohort_anchor(samples))
        g = 0
        keep = []
        for s in samples:
            for rg in s.read_groups:
                if pinned == "device":                          # arrays already resident on the GPU (pd_contig_push_device)
                    import torch
                    dp = torch.from_numpy(np.ascontiguousarray(rg.pos, dtype=np.uint32).view(np.int32)).to(f"cuda:{device}")
                    dd = torch.from_numpy(np.ascontiguousarray(rg.dev, dtype=np.int32)).to(f"cuda:{device}")
                    keep.append((dp, dd))
                    sc.push_device(g, dp.numel(), dp.data_ptr(), dd.data_ptr())
                elif pinned == "compact32":
                    sc.push_compact32(g, *[_page_locked(a) for a in compact32_encode(rg.pos, rg.dev)])
                elif pinned == "compact":
                    sc.push_compact(g, *[_page_locked(a) for a in compact_encode(rg.pos, rg.dev)])
                elif pinned:
                    sc.push_pinned(g, _page_locked(np.ascontiguousarray(rg.pos, dtype=np.uint32)),
                                   _page_locked(np.ascontiguousarray(rg.dev, dtype=np.int32)))
                else:
                    sc.push(g, rg.pos, rg.dev)
                g += 1
        return sc.scan(first_window, n_windows), rgs
    finally:
        sc.close()


def shard_unique_id() -> bytes:
    """ncclUniqueId for pd_shard_attach_nccl (make it on rank 0, broadcast it)."""
    buf = (C.c_uint8 * 128)()
    rc = load_library().pd_shard_unique_id(buf)
    if rc != 0:
        raise ScanError(f"pd_shard_unique_id failed ({rc}): libnccl.so.2 not loadable?")
    return bytes(buf)


def split_samples(n_samples: int, world: int):
    """Contiguous sample blocks per rank (sizes differ by at most one)."""
    base, extra = divmod(int(n_samples), int(world))
    return [base + (1 if r < extra else 0) for r in range(world)]


def cohort_headers(samples):
    return [[dict(name=rg.spec.name, median=rg.median, stddev=rg.stddev, read_length=rg.spec.read_length,
                  hist_start=rg.hist_start, hist_end=rg.hist_end, hist_counts=rg.hist_counts) for rg in s.read_groups] for s in samples]


def sample_shard_scanner(samples, params: CallParameters, world: int, rank: int, device: int = 0, contig_len: int = 0):
    """Rank `rank` of a sample-sharded in-memory cohort: a Scanner holding the rank's block of samples (split_samples), its
    read pairs pushed and the cohort's window range reserved, not yet attached. Returns (scanner, read groups of the whole
    cohort, samples per rank, minInitDelLengths of the whole cohort): what attach_nccl / pd_shard_attach_group take."""
    rgs = read_groups_from_headers(cohort_headers(samples), params)                 # parameters of the WHOLE cohort
    spr = split_samples(len(samples), world)
    mi = np.array([r.min_init_del_len for r in rgs], dtype=np.uint32)
    anchor = cohort_anchor(samples)
    if not contig_len:
        contig_len = max(int(rg.pos[-1]) + 25000 for s in samples for rg in s.read_groups if rg.pos.size)
    s0 = sum(spr[:rank])
    local = [ReadGroup(**{**g.__dict__, "sample": g.sample - s0}) for g in rgs if s0 <= g.sample < s0 + spr[rank]]
    sc = Scanner(params, local, spr[rank], device)
    sc.begin_contig(anchor)
    sc.reserve_windows((contig_len - anchor) // 30 + 2)
    gi = 0
    for s in samples[s0:s0 + spr[rank]]:
        for rg in s.read_groups:
            sc.push(gi, rg.pos, rg.dev)
            gi += 1
    return sc, rgs, spr, mi


class ShardGroup:
    """A sample-sharded in-memory cohort over `world` contexts of THIS process (pd_shard_attach_group; devices[r] = GPU of
    rank r, default all on GPU 0). scan() is the collective pd_shard_group_scan and may be repeated; scanners[r].set_unify
    changes what the next scan returns (the same settings on every rank)."""

    def __init__(self, samples, params: CallParameters, world: int, devices=None, contig_len: int = 0):
        self.lib = load_library()
        devices = list(devices) if devices is not None else [0] * world
        self.world, self.scanners = world, []
        try:
            for r in range(world):
                sc, self.rgs, self.spr, mi = sample_shard_scanner(samples, params, world, r, devices[r], contig_len)
                self.scanners.append(sc)
            self.ctxs = (C.c_void_p * world)(*[sc.ctx for sc in self.scanners])
            sprs = np.array(self.spr, dtype=np.uint32)
            infos = (PdShardInfo * world)(*[PdShardInfo(r, world, len(samples), mi.size, mi.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                        sprs.ctypes.data_as(C.POINTER(C.c_uint32))) for r in range(world)])
            self._check(self.lib.pd_shard_attach_group(self.ctxs, world, infos), "pd_shard_attach_group")
        except BaseException:
            self.close()
            raise

    def _check(self, rc, what):
        if rc != 0:
            raise ScanError(f"[{rc}] {what}: " + "; ".join(self.lib.pd_last_error(sc.ctx).decode() for sc in self.scanners))

    def set_unify(self, *args, **kw):
        """Scanner.set_unify on every rank."""
        for sc in self.scanners:
            sc.set_unify(*args, **kw)

    def scan(self, first_window: int = 0, n_windows: int = 0) -> dict:
        """The result of rank 0 with the per-sample rows of all ranks concatenated in cohort order; `parts` = every rank's
        own result. The ranks must agree on the calls (and significant windows)."""
        outs = (PdResult * self.world)()
        self._check(self.lib.pd_shard_group_scan(self.ctxs, self.world, int(first_window), int(n_windows), outs), "pd_shard_group_scan")
        parts = [sc._result_dict(outs[r]) for r, sc in enumerate(self.scanners)]
        for p in parts[1:]:
            assert np.array_equal(p["calls"], parts[0]["calls"]), "ranks disagree on the calls"
            assert (p["significant_windows"] is None) == (parts[0]["significant_windows"] is None)
            if p["significant_windows"] is not None:
                assert np.array_equal(p["significant_windows"], parts[0]["significant_windows"]), "ranks disagree on the significant windows"
        merged = dict(parts[0])
        merged["per_sample"] = np.concatenate([p["per_sample"] for p in parts], axis=1)
        merged["parts"] = parts
        return merged

    def close(self):
        for sc in self.scanners:
            sc.close()


def scan_cohort_sample_sharded(samples, params: CallParameters, world: int, devices=None, first_window: int = 0, n_windows: int = 0,
                               contig_len: int = 0, unify: dict = None):
    """Sample-sharded scan of an in-memory cohort with `world` contexts of THIS process (ShardGroup). Returns the combined
    result (calls of rank 0, per-sample rows concatenated in cohort order) and the read groups of the whole cohort: window
    calls, or -- with unify=dict(mean_stddev=..., min_relative_window_cover=..., output_failed=...) -- the merged variants,
    the same on every rank, with the allele frequency over the whole cohort."""
    g = ShardGroup(samples, params, world, devices, contig_len)
    try:
        if unify:
            g.set_unify(**unify)
        return g.scan(first_window, n_windows), g.rgs
    finally:
        g.close()
