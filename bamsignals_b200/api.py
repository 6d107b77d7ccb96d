"""Host-side mirror of the bamsignals R interface for the counting path, on top of libbamsignals_cuda.so.

R is not installable offline, so the reference's R layer (R/wrappers.R, R/zzzCountSignals.R) is mirrored here in
Python with the same names, argument meaning, defaults and error behaviour; the compute goes through the C ABI of
include/bamsignals_cuda.h exactly as the R shim (rshim/, INTEGRATION.md) would.  There is no CPU fallback: if the
CUDA library is missing or no GPU is present the calls raise.

  bamCount / bamProfile / bamCoverage    R/wrappers.R:106-173
  pileup_core / coverage_core            R/RcppExports.R:12-18 (.Call boundary, src/bamsignals.cpp:444,474)
  flagMask / tlenFilter helpers          R/wrappers.R:76-98
  CountSignals                           R/zzzCountSignals.R:27-113
  GRanges                                the slots parseRegions reads (src/bamsignals.cpp:92-135)

Results on the GPU (beyond the R interface): `device=` on bamCount / bamProfile / bamCoverage, and `out=` (any int32
device array with __cuda_array_interface__) on pileup_core / coverage_core / Stage, count straight into device memory
through the bsg_*_device entry points; nothing of the result crosses PCIe.  torch is imported only for those.

Coverage as runs (beyond the R interface): `bamCoverage(..., runs=True)`, `coverage_runs_core` and
`Stage.coverage_runs` return a CoverageRuns - run-length (length, value) pairs per region, counted on the GPU through
bsg_coverage_runs, on the host or (device=) in torch tensors.  Profiles likewise: `bamProfile(..., runs=True)`,
`profile_runs_core` and `Stage.profile_runs` return a ProfileRuns (bsg_profile_runs), runs over bins per region and
strand row.

Strand-specific coverage (beyond the R interface): `ss=True` on bamCoverage, coverage_core, coverage_runs_core,
Stage.coverage and Stage.coverage_runs counts sense and antisense coverage in one pass (bsg_coverage_ss*).
"""
from __future__ import annotations

import ctypes as C
import os
import sys
import warnings
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

_LIB_PATH = os.environ.get("BSG_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libbamsignals_cuda.so")
_lib = None


class BamsignalsError(RuntimeError):
    """Raised for any non-zero return of the C ABI; .code holds the BSG_E* value."""

    def __init__(self, code, msg):
        super().__init__(msg)
        self.code = code


# ------------------------------------------------------------------------------------------------------------------
# GRanges: just the slots the native code reads (ranges@start/width, seqnames, strand)
# ------------------------------------------------------------------------------------------------------------------
class GRanges:
    """Minimal stand-in for GenomicRanges::GRanges: seqnames, 1-based start, width, strand in {'+','-','*'}."""

    def __init__(self, seqnames: Sequence[str], start: Sequence[int], width: Sequence[int],
                 strand: Optional[Sequence[str]] = None, seqlevels: Optional[Sequence[str]] = None):
        n = len(start)
        if len(seqnames) != n or len(width) != n:
            raise ValueError("seqnames, start and width must have the same length")
        seqnames = [str(s) for s in seqnames]
        if seqlevels is None:
            seqlevels = list(dict.fromkeys(seqnames))
        self.seqlevels = [str(s) for s in seqlevels]
        lut = {s: i for i, s in enumerate(self.seqlevels)}
        try:
            self.seq_idx = np.fromiter((lut[s] for s in seqnames), dtype=np.int32, count=n)
        except KeyError as e:
            raise ValueError(f"seqname {e} not in seqlevels") from None
        self.start = np.ascontiguousarray(start, dtype=np.int32)
        self.width = np.ascontiguousarray(width, dtype=np.int32)
        if (self.width < 0).any():
            raise ValueError("negative widths are not allowed")
        if strand is None:
            self.strand = np.zeros(n, dtype=np.int8)
        elif isinstance(strand, np.ndarray) and strand.dtype == np.int8:
            self.strand = np.ascontiguousarray(strand)
        else:
            self.strand = np.fromiter(((1 if s == "+" else -1 if s == "-" else 0) for s in strand), dtype=np.int8, count=n)

    @classmethod
    def from_codes(cls, seqlevels, seq_idx, start, width, strand_i8):
        """Vectorised constructor for large region sets (no per-element Python work)."""
        self = cls.__new__(cls)
        self.seqlevels = [str(s) for s in seqlevels]
        self.seq_idx = np.ascontiguousarray(seq_idx, dtype=np.int32)
        self.start = np.ascontiguousarray(start, dtype=np.int32)
        self.width = np.ascontiguousarray(width, dtype=np.int32)
        self.strand = np.ascontiguousarray(strand_i8, dtype=np.int8)
        return self

    def __len__(self):
        return len(self.start)

    def __getitem__(self, idx):
        idx = np.arange(len(self))[idx]
        return GRanges.from_codes(self.seqlevels, self.seq_idx[idx], self.start[idx], self.width[idx], self.strand[idx])

    @property
    def seqnames(self):
        return [self.seqlevels[i] for i in self.seq_idx]


# ------------------------------------------------------------------------------------------------------------------
# CountSignals container (R/zzzCountSignals.R)
# ------------------------------------------------------------------------------------------------------------------
def _is_tensor(x):
    torch = sys.modules.get("torch")            # a tensor exists only if torch was imported: never import it here
    return torch is not None and isinstance(x, torch.Tensor)


def _pairs(v):
    """(2, w) view [sense; antisense] of an interleaved slice [s_0, a_0, s_1, ...]: R's IntegerMatrix(2, w) memory order."""
    return v.view(-1, 2).t() if _is_tensor(v) else v.reshape((2, -1), order="F")


def _permute(a, axes):
    return a.permute(*axes) if _is_tensor(a) else a.transpose(axes)


class CountSignals:
    """List-like container: signal i is a (w,) int32 vector, or a (2, w) matrix [sense; antisense] when ss.

    The (2, w) matrices are Fortran-ordered views into the flat result buffer, i.e. the memory layout of R's
    IntegerMatrix(2, w) (src/bamsignals.cpp:178-181): [sense_0, antisense_0, sense_1, ...].  When built from the
    library's flat result (`flat` + `offsets`) the per-region views are created on first use.  `flat` may be a torch
    tensor (device=): the views, alignSignals and as_list are then tensors of the same shapes and element order."""

    rownames = ("sense", "antisense")

    def __init__(self, signals: Optional[List[np.ndarray]], ss: bool, flat: Optional[np.ndarray] = None,
                 offsets: Optional[np.ndarray] = None):
        self.ss = bool(ss)
        self._signals = signals
        self._flat, self._offsets = flat, offsets
        if signals is not None:
            for s in signals:                                # checkList, src/CountSignals.cpp:4-16
                if self.ss and not (s.ndim == 2 and s.shape[0] == 2):
                    raise ValueError("strand-specific signals must be matrices with two rows")
                if not self.ss and s.ndim != 1:
                    raise ValueError("signals must be vectors")

    def _view(self, i):
        v = self._flat[int(self._offsets[i]):int(self._offsets[i + 1])]
        return _pairs(v) if self.ss else v

    @property
    def signals(self):
        if self._signals is None:
            self._signals = [self._view(i) for i in range(len(self._offsets) - 1)]
        return self._signals

    def __len__(self):                                       # R/zzzCountSignals.R:46
        return len(self._signals) if self._signals is not None else len(self._offsets) - 1

    def width(self):                                         # R/zzzCountSignals.R:54-56 (fastWidth)
        if self._signals is None:
            return np.diff(self._offsets) // (2 if self.ss else 1)
        return np.array([s.shape[-1] for s in self._signals], dtype=np.int64)

    def __getitem__(self, i):                                # R/zzzCountSignals.R:68-77
        if isinstance(i, (int, np.integer)):
            if i < 0 or i >= len(self):
                raise IndexError("subscript out of bounds")
            return self._signals[i] if self._signals is not None else self._view(int(i))
        idx = np.arange(len(self))[i]
        return CountSignals([self[int(k)] for k in idx], self.ss)

    def as_list(self):                                       # R/zzzCountSignals.R:83-96
        return list(self.signals)

    def alignSignals(self):                                  # R/zzzCountSignals.R:107-113
        w = self.width()
        if len(w) and (w != w[0]).any():
            raise ValueError("all signals must have the same width")
        if len(self) == 0:
            return self._flat.new_zeros((0,)) if _is_tensor(self._flat) else np.zeros((0,), dtype=np.int32)
        if self._signals is None:                            # contiguous result: one reshape, no copies
            R, w0 = len(self), int(w[0])
            if not self.ss:
                return _permute(self._flat.reshape((R, w0)), (1, 0))
            return _permute(self._flat.reshape((R, w0, 2)), (2, 1, 0))
        if _is_tensor(self._signals[0]):
            return sys.modules["torch"].stack(self._signals, dim=-1)
        return np.stack(self._signals, axis=-1)              # [w, R] or [2, w, R] like simplify2array

    def __repr__(self):
        kind = "strand-specific" if self.ss else "strand-unspecific"
        return f"CountSignals object with {len(self)} {kind} signals"


def _expand_runs(lengths, values, offsets):
    """The dense vector that runs describe (every list's expansion, one after another, on the runs' device) and the
    dense offset of every list (numpy int64, len(offsets))."""
    if _is_tensor(lengths):
        torch = sys.modules["torch"]
        lengths = lengths.long()
        flat = torch.repeat_interleave(values, lengths)
        ends = torch.zeros(len(lengths) + 1, dtype=torch.int64, device=lengths.device)
        torch.cumsum(lengths, 0, out=ends[1:])
        return flat, ends[torch.from_numpy(offsets).to(lengths.device)].cpu().numpy()
    flat = np.repeat(values, lengths)
    ends = np.zeros(len(lengths) + 1, dtype=np.int64)
    np.cumsum(lengths, out=ends[1:])
    return flat, ends[offsets]


class _RunLists:
    """Flat int32 `lengths` / `values` (numpy arrays or torch tensors on one device) and numpy int64 `offsets`: list k
    is lengths[offsets[k]:offsets[k+1]] elements of values[offsets[k]:offsets[k+1]].  Without `ss` list i is region i;
    with `ss` list 2i is region i's sense row and list 2i+1 its antisense row.  len() is R; [i] is (lengths, values), or
    with ss a (sense, antisense) pair of them."""

    def __init__(self, lengths, values, offsets, ss=False):
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        if offsets.ndim != 1 or len(offsets) < 1 or offsets[0] != 0 or (np.diff(offsets) < 0).any():
            raise ValueError("offsets must be a non-decreasing int64 vector that starts at 0")
        if len(lengths) != offsets[-1] or len(values) != offsets[-1]:
            raise ValueError(f"lengths and values must have offsets[-1] = {int(offsets[-1])} elements")
        self.lengths, self.values, self.offsets = lengths, values, offsets
        self.ss = bool(ss)
        if self.ss and (len(self.offsets) - 1) % 2:
            raise ValueError("a strand-specific result has two lists per region: offsets must have 2R + 1 entries")

    def __len__(self):
        return (len(self.offsets) - 1) // (2 if self.ss else 1)

    def __getitem__(self, i):
        i = self._index(i)
        return (self._list(2 * i), self._list(2 * i + 1)) if self.ss else self._list(i)

    def _list(self, k):
        a, b = int(self.offsets[k]), int(self.offsets[k + 1])
        return self.lengths[a:b], self.values[a:b]

    def _index(self, i):
        if not isinstance(i, (int, np.integer)):
            raise TypeError(f"{type(self).__name__} indices must be integers")
        if i < 0 or i >= len(self):
            raise IndexError("subscript out of bounds")
        return int(i)

    def to_dense(self) -> CountSignals:
        """The dense result these runs describe (a CountSignals over one flat buffer on the runs' device, with the
        (2, w) [sense; antisense] views when ss)."""
        if not self.ss:
            flat, dense_off = _expand_runs(self.lengths, self.values, self.offsets)
            return CountSignals(None, False, flat=flat, offsets=dense_off)
        # Every region's dense slice [s_0, a_0, s_1, ...] starts at an even offset, so the even elements of the whole
        # result are all sense rows one after another and the odd ones all antisense rows.
        sizes = np.diff(self.offsets)
        row_of_run = np.repeat(np.arange(len(sizes)) % 2, sizes)
        rows = []
        for a in (0, 1):
            sel = row_of_run == a
            if _is_tensor(self.lengths):
                sel = sys.modules["torch"].from_numpy(sel).to(self.lengths.device)
            off = np.zeros(len(self) + 1, dtype=np.int64)
            np.cumsum(sizes[a::2], out=off[1:])
            rows.append(_expand_runs(self.lengths[sel], self.values[sel], off))
        (sense, bins), (anti, bins_anti) = rows
        if not np.array_equal(bins, bins_anti):
            raise ValueError("the sense and antisense rows of a region must have the same number of bins")
        if _is_tensor(sense):
            flat = sys.modules["torch"].stack((sense, anti), dim=1).reshape(-1)
        else:
            flat = np.empty(2 * len(sense), dtype=sense.dtype)
            flat[0::2], flat[1::2] = sense, anti
        return CountSignals(None, True, flat=flat, offsets=2 * bins)


class CoverageRuns(_RunLists):
    """bamCoverage as runs: region i's coverage (in region orientation) is lengths[offsets[i]:offsets[i+1]] bases of
    values[offsets[i]:offsets[i+1]].  `lengths` / `values` are flat int32 numpy arrays or torch tensors on one device;
    `offsets` is numpy int64 (R + 1).  Adjacent runs of a region differ in value, every length is >= 1, a zero-width
    region has no runs.  The same thing as an RleList of GenomicAlignments::coverage, one Rle per region.
    With `ss` (strand-specific coverage) the lists are those of a strand-specific ProfileRuns: list 2i is region i's
    sense row, list 2i+1 its antisense row, `offsets` has 2R + 1 entries, [i] is the (sense, antisense) pair and
    to_dense() gives bamCoverage(..., ss=True)'s CountSignals."""

    def __init__(self, lengths, values, offsets, ss=False):
        super().__init__(lengths, values, offsets, ss)

    def __repr__(self):
        if self.ss:
            return f"CoverageRuns object with {len(self)} strand-specific regions and {int(self.offsets[-1])} runs"
        return f"CoverageRuns object with {len(self)} regions and {int(self.offsets[-1])} runs"


class ProfileRuns(_RunLists):
    """bamProfile as runs over bins (in region orientation, a partial last bin is one element).  Without `ss` list i is
    region i's profile; with `ss` list 2i is region i's sense row and list 2i+1 its antisense row, so `offsets` has
    (ss ? 2R : R) + 1 entries.  Adjacent runs of a list differ in value, every length is >= 1, a list's lengths sum to
    its bin count, a zero-width region has no runs.  len() is R; [i] is (lengths, values), or with ss a
    (sense, antisense) pair of them."""

    def __init__(self, lengths, values, offsets, ss):
        super().__init__(lengths, values, offsets, ss)

    def __repr__(self):
        kind = "strand-specific" if self.ss else "strand-unspecific"
        return f"ProfileRuns object with {len(self)} {kind} regions and {int(self.offsets[-1])} runs"


# ------------------------------------------------------------------------------------------------------------------
# argument helpers (R/wrappers.R:76-98)
# ------------------------------------------------------------------------------------------------------------------
def flagMask(paired_end: str) -> int:
    return 66 if paired_end != "ignore" else 0


def _match_arg(value, choices):
    if isinstance(value, (tuple, list)):
        value = value[0]
    if value not in choices:
        raise ValueError(f"'arg' should be one of {', '.join(repr(c) for c in choices)}")
    return value


@dataclass
class Marshalled:
    """ctypes views of a GRanges for the C ABI (kept alive by this object)."""
    R: int
    levels: C.Array
    n_levels: int
    seq_idx: np.ndarray
    loc: np.ndarray
    width: np.ndarray
    strand: np.ndarray


def marshal_regions(gr: GRanges) -> Marshalled:
    if not isinstance(gr, GRanges):
        raise TypeError("must provide a GRanges object")             # src/bamsignals.cpp:94
    levels = (C.c_char_p * max(1, len(gr.seqlevels)))(*[s.encode() for s in gr.seqlevels])
    loc = np.ascontiguousarray(gr.start - 1, dtype=np.int32)         # 1-based -> 0-based, src/bamsignals.cpp:131
    return Marshalled(len(gr), levels, len(gr.seqlevels), gr.seq_idx, loc, gr.width, gr.strand)


def output_layout(width: np.ndarray, binsize: int, ss: bool):
    """Offsets (int64, R+1) of every region's slice in the flat result buffer (allocateList, :139-192)."""
    mult = 2 if ss else 1
    if binsize <= 0:
        per = np.full(len(width), mult, dtype=np.int64)
    else:
        per = mult * ((width.astype(np.int64) + binsize - 1) // binsize)
    off = np.zeros(len(width) + 1, dtype=np.int64)
    np.cumsum(per, out=off[1:])
    return off


def split_signals(flat: np.ndarray, offsets: np.ndarray, ss: bool):
    """Zero-copy per-region views shaped like the R list elements."""
    if ss:
        return [flat[offsets[i]:offsets[i + 1]].reshape((2, -1), order="F") for i in range(len(offsets) - 1)]
    return [flat[offsets[i]:offsets[i + 1]] for i in range(len(offsets) - 1)]


def _p(a, ty):
    return a.ctypes.data_as(C.POINTER(ty))


# ------------------------------------------------------------------------------------------------------------------
# the native library
# ------------------------------------------------------------------------------------------------------------------
class BsgOpts(C.Structure):
    _fields_ = [("struct_size", C.c_int32), ("n_devices", C.c_int32), ("devices", C.c_int32 * 16),
                ("inflate_threads", C.c_int32), ("batch_bytes", C.c_int64), ("verify_crc", C.c_int32),
                ("use_cache", C.c_int32), ("gpu_inflate", C.c_int32), ("stream_min_ints", C.c_int32),
                ("result_pack", C.c_int32), ("walk_scheme", C.c_int32),
                ("resident_scheme", C.c_int32), ("reserved", C.c_int32 * 4)]


class BsgTimings(C.Structure):
    _fields_ = [("records", C.c_int64), ("records_kept", C.c_int64), ("bytes_compressed", C.c_int64),
                ("bytes_inflated", C.c_int64), ("candidates", C.c_int64), ("out_elems", C.c_int64),
                ("n_tiles", C.c_int64), ("n_batches", C.c_int64), ("n_launches", C.c_int64),
                ("n_devices", C.c_int32), ("upload_mode", C.c_int32),
                ("ms_total", C.c_double), ("ms_plan", C.c_double), ("ms_fetch", C.c_double),
                ("ms_h2d", C.c_double), ("ms_d2h", C.c_double),
                ("ms_decode", C.c_double), ("ms_filter", C.c_double), ("ms_join", C.c_double),
                ("ms_count", C.c_double), ("ms_inflate_gpu", C.c_double), ("ms_kernels", C.c_double),
                ("ms_device", C.c_double), ("bytes_d2h", C.c_double), ("reserved", C.c_double * 6)]


def lib():
    """Load libbamsignals_cuda.so (built in-tree by __graft_entry__.build()); fail loudly if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise ImportError(f"{_LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`. "
                          "There is no CPU fallback for the counting path.")
    L = C.CDLL(_LIB_PATH)
    i32p, i64p, i8p = C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_int8)
    region_args = [C.c_char_p, C.c_int64, C.POINTER(C.c_char_p), C.c_int32, i32p, i32p, i32p, i8p]
    L.bsg_pileup.argtypes = region_args + [i32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                           C.c_int32, C.c_int32, i32p, i64p, C.POINTER(C.POINTER(C.c_int32)),
                                           C.POINTER(BsgOpts)]
    L.bsg_pileup.restype = C.c_int
    L.bsg_coverage.argtypes = region_args + [i32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                             i32p, i64p, C.POINTER(C.POINTER(C.c_int32)), C.POINTER(BsgOpts)]
    L.bsg_coverage.restype = C.c_int
    L.bsg_pileup_device.argtypes = region_args + [i32p] + [C.c_int32] * 8 + [C.c_void_p, i64p, C.c_void_p, C.POINTER(BsgOpts)]
    L.bsg_pileup_device.restype = C.c_int
    L.bsg_coverage_device.argtypes = region_args + [i32p] + [C.c_int32] * 5 + [C.c_void_p, i64p, C.c_void_p, C.POINTER(BsgOpts)]
    L.bsg_coverage_device.restype = C.c_int
    L.bsg_last_error.restype = C.c_char_p
    L.bsg_version.restype = C.c_char_p
    L.bsg_get_timings.argtypes = [C.POINTER(BsgTimings)]
    L.bsg_get_timings.restype = C.c_int
    L.bsg_shutdown.restype = None
    L.bsg_output_layout.argtypes = [C.c_int64, i32p, C.c_int32, C.c_int32, i64p]
    L.bsg_output_layout.restype = C.c_int64
    L.bsg_device_count.restype = C.c_int
    L.bsg_stage_open.argtypes = [C.POINTER(C.c_void_p)] + region_args + [C.c_int32, C.POINTER(BsgOpts)]
    L.bsg_stage_open.restype = C.c_int
    L.bsg_pileup_staged.argtypes = [C.c_void_p, i32p] + [C.c_int32] * 7 + [i32p, i64p]
    L.bsg_pileup_staged.restype = C.c_int
    L.bsg_coverage_staged.argtypes = [C.c_void_p, i32p] + [C.c_int32] * 4 + [i32p, i64p]
    L.bsg_coverage_staged.restype = C.c_int
    L.bsg_pileup_staged_device.argtypes = [C.c_void_p, i32p] + [C.c_int32] * 7 + [C.c_void_p, i64p, C.c_void_p]
    L.bsg_pileup_staged_device.restype = C.c_int
    L.bsg_coverage_staged_device.argtypes = [C.c_void_p, i32p] + [C.c_int32] * 4 + [C.c_void_p, i64p, C.c_void_p]
    L.bsg_coverage_staged_device.restype = C.c_int
    L.bsg_coverage_runs.argtypes = region_args + [i32p] + [C.c_int32] * 5 + [i64p, C.POINTER(C.c_void_p), C.POINTER(BsgOpts)]
    L.bsg_coverage_runs.restype = C.c_int
    L.bsg_coverage_runs_staged.argtypes = [C.c_void_p, i32p] + [C.c_int32] * 4 + [i64p, C.POINTER(C.c_void_p)]
    L.bsg_coverage_runs_staged.restype = C.c_int
    L.bsg_profile_runs.argtypes = region_args + [i32p] + [C.c_int32] * 8 + [i64p, C.POINTER(C.c_void_p), C.POINTER(BsgOpts)]
    L.bsg_profile_runs.restype = C.c_int
    L.bsg_profile_runs_staged.argtypes = [C.c_void_p, i32p] + [C.c_int32] * 7 + [i64p, C.POINTER(C.c_void_p)]
    L.bsg_profile_runs_staged.restype = C.c_int
    L.bsg_coverage_ss.argtypes = region_args + [i32p] + [C.c_int32] * 6 + [i32p, i64p, C.POINTER(C.POINTER(C.c_int32)),
                                                                       C.POINTER(BsgOpts)]
    L.bsg_coverage_ss.restype = C.c_int
    L.bsg_coverage_ss_device.argtypes = region_args + [i32p] + [C.c_int32] * 6 + [C.c_void_p, i64p, C.c_void_p, C.POINTER(BsgOpts)]
    L.bsg_coverage_ss_device.restype = C.c_int
    L.bsg_coverage_ss_staged.argtypes = [C.c_void_p, i32p] + [C.c_int32] * 5 + [i32p, i64p]
    L.bsg_coverage_ss_staged.restype = C.c_int
    L.bsg_coverage_ss_staged_device.argtypes = [C.c_void_p, i32p] + [C.c_int32] * 5 + [C.c_void_p, i64p, C.c_void_p]
    L.bsg_coverage_ss_staged_device.restype = C.c_int
    L.bsg_coverage_runs_ss.argtypes = region_args + [i32p] + [C.c_int32] * 6 + [i64p, C.POINTER(C.c_void_p), C.POINTER(BsgOpts)]
    L.bsg_coverage_runs_ss.restype = C.c_int
    L.bsg_coverage_runs_ss_staged.argtypes = [C.c_void_p, i32p] + [C.c_int32] * 5 + [i64p, C.POINTER(C.c_void_p)]
    L.bsg_coverage_runs_ss_staged.restype = C.c_int
    L.bsg_runs_read.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.bsg_runs_read.restype = C.c_int
    L.bsg_runs_free.argtypes = [C.c_void_p]
    L.bsg_runs_free.restype = None
    L.bsg_stage_view.argtypes = [C.POINTER(C.c_void_p), C.c_void_p] + region_args[1:]
    L.bsg_stage_view.restype = C.c_int
    L.bsg_stage_close.argtypes = [C.c_void_p]
    L.bsg_stage_close.restype = None
    L.bsg_debug_plan.argtypes = region_args + [C.c_int64, i64p, i64p, i64p, i32p, i32p, C.c_int64]
    L.bsg_debug_plan.restype = C.c_int64
    L.bsg_write_sam_as_bam_and_index.argtypes = [C.c_char_p, C.c_char_p]
    L.bsg_write_sam_as_bam_and_index.restype = C.c_int
    _lib = L
    return L


def _check(rc):
    if rc != 0:
        raise BamsignalsError(rc, lib().bsg_last_error().decode(errors="replace"))


def default_opts(**kw) -> BsgOpts:
    o = BsgOpts()
    o.struct_size = C.sizeof(BsgOpts)
    o.verify_crc = 1
    for k, v in kw.items():
        if k == "devices":
            o.n_devices = len(v)
            for i, d in enumerate(v):
                o.devices[i] = d
        else:
            setattr(o, k, v)
    return o


def debug_plan(bampath, gr, ext=0, cap=1 << 22) -> dict:
    """bsg_debug_plan: what the fetch planner decides for `gr` with halo `ext`, and the (tid, pos) of every record inside
    the planned ranges.  Host-only diagnostic (used by the CPU tests of the index logic); it counts nothing."""
    m = marshal_regions(gr)
    nseg, cb, ub = C.c_int64(), C.c_int64(), C.c_int64()
    tid, pos = np.empty(cap, dtype=np.int32), np.empty(cap, dtype=np.int32)
    n = lib().bsg_debug_plan(os.fsencode(bampath), m.R, m.levels, m.n_levels, _p(m.seq_idx, C.c_int32), _p(m.loc, C.c_int32),
                             _p(m.width, C.c_int32), _p(m.strand, C.c_int8), int(ext), C.byref(nseg), C.byref(cb), C.byref(ub),
                             _p(tid, C.c_int32), _p(pos, C.c_int32), cap)
    if n < 0:
        _check(int(n))
    if n > cap:
        return debug_plan(bampath, gr, ext, int(n))
    return dict(records=int(n), segments=nseg.value, bytes_compressed=cb.value, bytes_inflated=ub.value, tid=tid[:n], pos=pos[:n])


def writeSamAsBamAndIndex(sampath, bampath) -> bool:
    """bamsignals:::writeSamAsBamAndIndex (R/RcppExports.R:20-22, src/bamsignals.cpp:496-534): SAM text ->
    coordinate-sorted BAM + .bai.  Host-only."""
    _check(lib().bsg_write_sam_as_bam_and_index(os.fsencode(os.path.expanduser(sampath)), os.fsencode(os.path.expanduser(bampath))))
    return True


def timings() -> dict:
    t = BsgTimings()
    lib().bsg_get_timings(C.byref(t))
    return {f: getattr(t, f) for f, _ in BsgTimings._fields_ if f not in ("reserved", "pad")}


def device_buffer(out, total):
    """(pointer, stream) of a caller's device buffer for the bsg_*_device entry points.  `out` is anything with
    __cuda_array_interface__ (a torch CUDA tensor, a CuPy array): one-dimensional, int32, C-contiguous, at least `total`
    elements.  The stream is the one the library orders its writes after: torch's current stream for a tensor, else the
    interface's `stream` entry (0, the legacy default stream, when absent)."""
    if _is_tensor(out):
        import torch
        if not out.is_cuda:
            raise TypeError(f"out must be a CUDA tensor, not one on {out.device}")
        if out.dtype != torch.int32:
            raise TypeError(f"out must be an int32 tensor, not {out.dtype}")
        if out.dim() != 1:
            raise ValueError(f"out must be one-dimensional, not of shape {tuple(out.shape)}")
        if not out.is_contiguous():
            raise ValueError("out must be C-contiguous")
        if out.numel() < total:
            raise ValueError(f"out has {out.numel()} elements, the result needs {total}")
        return out.data_ptr(), torch.cuda.current_stream(out.device).cuda_stream
    try:
        cai = out.__cuda_array_interface__
    except (AttributeError, TypeError):
        raise TypeError("out must be a device array with __cuda_array_interface__ (a torch CUDA tensor, a CuPy array)") from None
    if np.dtype(cai["typestr"]) != np.int32:
        raise TypeError(f"out must be int32, not {np.dtype(cai['typestr'])}")
    shape = tuple(cai["shape"])
    if len(shape) != 1:
        raise ValueError(f"out must be one-dimensional, not of shape {shape}")
    strides = cai.get("strides")
    if strides is not None and shape[0] > 1 and tuple(strides) != (4,):
        raise ValueError("out must be C-contiguous")
    if shape[0] < total:
        raise ValueError(f"out has {shape[0]} elements, the result needs {total}")
    ptr, readonly = cai["data"]
    if readonly:
        raise ValueError("out is read-only")
    return ptr, cai.get("stream") or 0


def _cuda_device(device):
    """`device` (a torch.device, "cuda:1" or 1) as a torch.device with an index; TypeError unless it is a CUDA device."""
    import torch
    dev = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
    if dev.type != "cuda":
        raise TypeError(f"device must be a CUDA device, not {dev}")
    return dev if dev.index is not None else torch.device("cuda", torch.cuda.current_device())


def _empty_on(device, gr, binsize, ss):
    """The flat int32 result buffer of a call, allocated by torch on `device` (a torch.device, "cuda:1" or 1)."""
    import torch
    if not isinstance(gr, GRanges):
        raise TypeError("must provide a GRanges object")             # src/bamsignals.cpp:94
    dev = _cuda_device(device)
    n = int(output_layout(gr.width, int(binsize), bool(ss))[-1])
    return torch.empty(n, dtype=torch.int32, device=dev)


def pileup_core(bampath, gr, tlen_filter, mapqual=0, binsize=1, shift=0, ss=False, requiredF=0, filteredF=-1,
                pe_mid=False, maxgap=16385, opts: Optional[BsgOpts] = None, _lazy=False, out=None):
    """The .Call('bamsignals_pileup_core') entry point (src/bamsignals.cpp:444-461); binsize <= 0 means bamCount.
    Returns the R `List`: one flat vector / (2,R) matrix for bamCount, else one array per region.
    With `out` (a device array, see device_buffer) the flat result is written there on the GPU and `out` is returned."""
    m = marshal_regions(gr)
    off = output_layout(m.width, int(binsize), bool(ss))
    tl = None if tlen_filter is None else np.asarray(tlen_filter, dtype=np.int32)
    if out is not None:
        ptr, stream = device_buffer(out, int(off[-1]))
        _check(lib().bsg_pileup_device(os.fsencode(bampath), m.R, m.levels, m.n_levels, _p(m.seq_idx, C.c_int32),
                                       _p(m.loc, C.c_int32), _p(m.width, C.c_int32), _p(m.strand, C.c_int8),
                                       None if tl is None else _p(tl, C.c_int32), int(mapqual), int(binsize), int(shift),
                                       int(bool(ss)), int(requiredF), int(filteredF), int(bool(pe_mid)), int(maxgap),
                                       ptr, _p(off, C.c_int64), stream, None if opts is None else C.byref(opts)))
        return (out, off) if _lazy else out
    flat = np.empty(int(off[-1]), dtype=np.int32)
    rc = lib().bsg_pileup(os.fsencode(bampath), m.R, m.levels, m.n_levels, _p(m.seq_idx, C.c_int32),
                          _p(m.loc, C.c_int32), _p(m.width, C.c_int32), _p(m.strand, C.c_int8),
                          None if tl is None else _p(tl, C.c_int32), int(mapqual), int(binsize), int(shift),
                          int(bool(ss)), int(requiredF), int(filteredF), int(bool(pe_mid)), int(maxgap),
                          _p(flat, C.c_int32), _p(off, C.c_int64), None,
                          None if opts is None else C.byref(opts))
    _check(rc)
    if binsize <= 0:
        return [flat.reshape((2, -1), order="F") if ss else flat]
    if _lazy:
        return flat, off
    return split_signals(flat, off, bool(ss))


def coverage_core(bampath, gr, tlen_filter, mapqual=0, requiredF=0, filteredF=-1, tspan=False, maxgap=16385,
                  opts: Optional[BsgOpts] = None, _lazy=False, out=None, ss=False):
    """The .Call('bamsignals_coverage_core') entry point (src/bamsignals.cpp:474-494).  `out`: as for pileup_core.
    ss=True (beyond the reference): strand-specific coverage (bsg_coverage_ss), one (2, w) [sense; antisense] matrix per
    region, the layout of a binsize-1 strand-specific profile."""
    m = marshal_regions(gr)
    ss = bool(ss)
    off = output_layout(m.width, 1, ss)
    tl = None if tlen_filter is None else np.asarray(tlen_filter, dtype=np.int32)
    if out is not None:
        ptr, stream = device_buffer(out, int(off[-1]))
        _check(lib().bsg_coverage_ss_device(os.fsencode(bampath), m.R, m.levels, m.n_levels, _p(m.seq_idx, C.c_int32),
                                            _p(m.loc, C.c_int32), _p(m.width, C.c_int32), _p(m.strand, C.c_int8),
                                            None if tl is None else _p(tl, C.c_int32), int(mapqual), int(requiredF),
                                            int(filteredF), int(bool(tspan)), int(ss), int(maxgap), ptr, _p(off, C.c_int64),
                                            stream, None if opts is None else C.byref(opts)))
        return (out, off) if _lazy else out
    flat = np.empty(int(off[-1]), dtype=np.int32)
    rc = lib().bsg_coverage_ss(os.fsencode(bampath), m.R, m.levels, m.n_levels, _p(m.seq_idx, C.c_int32),
                               _p(m.loc, C.c_int32), _p(m.width, C.c_int32), _p(m.strand, C.c_int8),
                               None if tl is None else _p(tl, C.c_int32), int(mapqual), int(requiredF), int(filteredF),
                               int(bool(tspan)), int(ss), int(maxgap), _p(flat, C.c_int32), _p(off, C.c_int64), None,
                               None if opts is None else C.byref(opts))
    _check(rc)
    if _lazy:
        return flat, off
    return split_signals(flat, off, ss)


def _take_runs(h, offsets, device):
    """Copy a bsg_runs result into numpy arrays (device None) or torch tensors on `device`, then free it: (lengths,
    values)."""
    try:
        n = int(offsets[-1])
        if device is None:
            lengths, values = np.empty(n, dtype=np.int32), np.empty(n, dtype=np.int32)
            _check(lib().bsg_runs_read(h, lengths.ctypes.data or None, values.ctypes.data or None, None))
        else:
            import torch
            lengths = torch.empty(n, dtype=torch.int32, device=device)
            values = torch.empty(n, dtype=torch.int32, device=device)
            _check(lib().bsg_runs_read(h, lengths.data_ptr() or None, values.data_ptr() or None,
                                       torch.cuda.current_stream(device).cuda_stream))
    finally:
        lib().bsg_runs_free(h)
    return lengths, values


def coverage_runs_core(bampath, gr, tlen_filter, mapqual=0, requiredF=0, filteredF=-1, tspan=False, maxgap=16385,
                       opts: Optional[BsgOpts] = None, device=None, ss=False) -> CoverageRuns:
    """coverage_core's arguments -> the coverage as runs (bsg_coverage_runs_ss).  device=None: numpy arrays on the host;
    device= a CUDA device: torch tensors there (the call runs on that device; only the offsets cross PCIe)."""
    m = marshal_regions(gr)
    dev = None if device is None else _cuda_device(device)
    if dev is not None and opts is None:
        opts = default_opts(devices=[dev.index])
    tl = None if tlen_filter is None else np.asarray(tlen_filter, dtype=np.int32)
    offsets = np.zeros((2 if ss else 1) * m.R + 1, dtype=np.int64)
    h = C.c_void_p()
    _check(lib().bsg_coverage_runs_ss(os.fsencode(bampath), m.R, m.levels, m.n_levels, _p(m.seq_idx, C.c_int32),
                                      _p(m.loc, C.c_int32), _p(m.width, C.c_int32), _p(m.strand, C.c_int8),
                                      None if tl is None else _p(tl, C.c_int32), int(mapqual), int(requiredF),
                                      int(filteredF), int(bool(tspan)), int(bool(ss)), int(maxgap), _p(offsets, C.c_int64),
                                      C.byref(h), None if opts is None else C.byref(opts)))
    return CoverageRuns(*_take_runs(h, offsets, dev), offsets, ss)


def profile_runs_core(bampath, gr, tlen_filter, mapqual=0, binsize=1, shift=0, ss=False, requiredF=0, filteredF=-1,
                      pe_mid=False, maxgap=16385, opts: Optional[BsgOpts] = None, device=None) -> ProfileRuns:
    """pileup_core's arguments (binsize >= 1) -> the profile as runs (bsg_profile_runs).  device=None: numpy arrays on
    the host; device= a CUDA device: torch tensors there (the call runs on that device; only the offsets cross PCIe)."""
    m = marshal_regions(gr)
    dev = None if device is None else _cuda_device(device)
    if dev is not None and opts is None:
        opts = default_opts(devices=[dev.index])
    tl = None if tlen_filter is None else np.asarray(tlen_filter, dtype=np.int32)
    offsets = np.zeros((2 if ss else 1) * m.R + 1, dtype=np.int64)
    h = C.c_void_p()
    _check(lib().bsg_profile_runs(os.fsencode(bampath), m.R, m.levels, m.n_levels, _p(m.seq_idx, C.c_int32),
                                  _p(m.loc, C.c_int32), _p(m.width, C.c_int32), _p(m.strand, C.c_int8),
                                  None if tl is None else _p(tl, C.c_int32), int(mapqual), int(binsize), int(shift),
                                  int(bool(ss)), int(requiredF), int(filteredF), int(bool(pe_mid)), int(maxgap),
                                  _p(offsets, C.c_int64), C.byref(h), None if opts is None else C.byref(opts)))
    return ProfileRuns(*_take_runs(h, offsets, dev), offsets, ss)


class Stage:
    """Resident session (bsg_stage_*): the byte ranges `gr` needs (with halo `ext_hint`) are fetched, inflated and
    uploaded once; every pileup()/coverage() call then runs the device path only.  want_output=False leaves the
    result in HBM (kernel-only timing); `out` (a device array, see device_buffer) receives it on the GPU and is
    returned."""

    def __init__(self, bampath, gr, ext_hint=0, opts: Optional[BsgOpts] = None):
        self._m = marshal_regions(gr)
        self._h = C.c_void_p()
        m = self._m
        _check(lib().bsg_stage_open(C.byref(self._h), os.fsencode(bampath), m.R, m.levels, m.n_levels,
                                    _p(m.seq_idx, C.c_int32), _p(m.loc, C.c_int32), _p(m.width, C.c_int32),
                                    _p(m.strand, C.c_int8), int(ext_hint), None if opts is None else C.byref(opts)))

    def pileup(self, tlen_filter, mapqual=0, binsize=1, shift=0, ss=False, requiredF=0, filteredF=-1, pe_mid=False,
               want_output=True, out=None):
        off = output_layout(self._m.width, int(binsize), bool(ss))
        tl = None if tlen_filter is None else np.asarray(tlen_filter, dtype=np.int32)
        if out is not None:
            ptr, stream = device_buffer(out, int(off[-1]))
            _check(lib().bsg_pileup_staged_device(self._h, None if tl is None else _p(tl, C.c_int32), int(mapqual),
                                                  int(binsize), int(shift), int(bool(ss)), int(requiredF), int(filteredF),
                                                  int(bool(pe_mid)), ptr, _p(off, C.c_int64), stream))
            return out
        flat = np.empty(int(off[-1]), dtype=np.int32) if want_output else None
        _check(lib().bsg_pileup_staged(self._h, None if tl is None else _p(tl, C.c_int32), int(mapqual), int(binsize),
                                       int(shift), int(bool(ss)), int(requiredF), int(filteredF), int(bool(pe_mid)),
                                       None if flat is None else _p(flat, C.c_int32), _p(off, C.c_int64)))
        return flat

    def coverage(self, tlen_filter, mapqual=0, requiredF=0, filteredF=-1, tspan=False, want_output=True, out=None, ss=False):
        """ss=True: strand-specific coverage, the flat interleaved layout of a binsize-1 strand-specific profile."""
        off = output_layout(self._m.width, 1, bool(ss))
        tl = None if tlen_filter is None else np.asarray(tlen_filter, dtype=np.int32)
        if out is not None:
            ptr, stream = device_buffer(out, int(off[-1]))
            _check(lib().bsg_coverage_ss_staged_device(self._h, None if tl is None else _p(tl, C.c_int32), int(mapqual),
                                                       int(requiredF), int(filteredF), int(bool(tspan)), int(bool(ss)), ptr,
                                                       _p(off, C.c_int64), stream))
            return out
        flat = np.empty(int(off[-1]), dtype=np.int32) if want_output else None
        _check(lib().bsg_coverage_ss_staged(self._h, None if tl is None else _p(tl, C.c_int32), int(mapqual),
                                            int(requiredF), int(filteredF), int(bool(tspan)), int(bool(ss)),
                                            None if flat is None else _p(flat, C.c_int32), _p(off, C.c_int64)))
        return flat

    def coverage_runs(self, tlen_filter, mapqual=0, requiredF=0, filteredF=-1, tspan=False, device=None,
                      ss=False) -> CoverageRuns:
        """coverage() as runs (bsg_coverage_runs_ss_staged); device= must be the session's device."""
        dev = None if device is None else _cuda_device(device)
        tl = None if tlen_filter is None else np.asarray(tlen_filter, dtype=np.int32)
        offsets = np.zeros((2 if ss else 1) * self._m.R + 1, dtype=np.int64)
        h = C.c_void_p()
        _check(lib().bsg_coverage_runs_ss_staged(self._h, None if tl is None else _p(tl, C.c_int32), int(mapqual),
                                                 int(requiredF), int(filteredF), int(bool(tspan)), int(bool(ss)),
                                                 _p(offsets, C.c_int64), C.byref(h)))
        return CoverageRuns(*_take_runs(h, offsets, dev), offsets, ss)

    def profile_runs(self, tlen_filter, mapqual=0, binsize=1, shift=0, ss=False, requiredF=0, filteredF=-1, pe_mid=False,
                     device=None) -> ProfileRuns:
        """pileup() (binsize >= 1) as runs (bsg_profile_runs_staged); device= must be the session's device."""
        dev = None if device is None else _cuda_device(device)
        tl = None if tlen_filter is None else np.asarray(tlen_filter, dtype=np.int32)
        offsets = np.zeros((2 if ss else 1) * self._m.R + 1, dtype=np.int64)
        h = C.c_void_p()
        _check(lib().bsg_profile_runs_staged(self._h, None if tl is None else _p(tl, C.c_int32), int(mapqual), int(binsize),
                                             int(shift), int(bool(ss)), int(requiredF), int(filteredF), int(bool(pe_mid)),
                                             _p(offsets, C.c_int64), C.byref(h)))
        return ProfileRuns(*_take_runs(h, offsets, dev), offsets, ss)

    def view(self, gr) -> "Stage":
        """The same resident records, counted over another region set (bsg_stage_view): no BAM bytes are read again.
        The returned Stage has every method of this one, with its layouts from `gr`, and this session's options and
        device.  A region outside what the session fetched is refused (BamsignalsError), as is a later call that needs
        more halo around `gr` than the session's index queries cover.  Closing this session first leaves the view usable."""
        m = marshal_regions(gr)
        v = Stage.__new__(Stage)
        v._m, v._h = m, C.c_void_p()
        _check(lib().bsg_stage_view(C.byref(v._h), self._h, m.R, m.levels, m.n_levels, _p(m.seq_idx, C.c_int32),
                                    _p(m.loc, C.c_int32), _p(m.width, C.c_int32), _p(m.strand, C.c_int8)))
        return v

    def close(self):
        if self._h:
            lib().bsg_stage_close(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def core_args(fn, **kw):
    """R-level keyword arguments of bamCount / bamProfile / bamCoverage -> the arguments of the native entry point
    (R/wrappers.R:112-116, :143-147, :165-169)."""
    if fn == "bamCoverage":
        pe = _match_arg(kw.get("paired_end", "ignore"), ("ignore", "extend"))
        return dict(tlen_filter=_tlen(kw.get("tlenFilter"), pe), mapqual=_trunc(kw.get("mapqual", 0)),
                    requiredF=flagMask(pe), filteredF=_trunc(kw.get("filteredFlag", -1)), tspan=pe == "extend")
    pe = _match_arg(kw.get("paired_end", "ignore"), ("ignore", "filter", "midpoint"))
    return dict(tlen_filter=_tlen(kw.get("tlenFilter"), pe), mapqual=_trunc(kw.get("mapqual", 0)),
                binsize=-1 if fn == "bamCount" else _trunc(kw.get("binsize", 1)), shift=_trunc(kw.get("shift", 0)),
                ss=bool(kw.get("ss", False)), requiredF=flagMask(pe), filteredF=_trunc(kw.get("filteredFlag", -1)),
                pe_mid=pe == "midpoint")


# ------------------------------------------------------------------------------------------------------------------
# the user-facing functions (R/wrappers.R:106-173)
# ------------------------------------------------------------------------------------------------------------------
def _trunc(x):
    return int(x)          # Rcpp's input_parameter<int> truncates R doubles


# device=None: host numpy results (the R interface).  device= a torch device ("cuda:1", 1, torch.device): the result is
# counted into a torch int32 tensor on that device (bsg_*_device) and stays there.
def bamCount(bampath, gr, mapqual=0, shift=0, ss=False, paired_end=("ignore", "filter", "midpoint"),
             tlenFilter=None, filteredFlag=-1, verbose=False, opts=None, device=None):
    pe = _match_arg(paired_end, ("ignore", "filter", "midpoint"))
    bampath = os.path.expanduser(bampath)
    out = None if device is None else _empty_on(device, gr, -1, ss)
    pu = pileup_core(bampath, gr, _tlen(tlenFilter, pe), _trunc(mapqual), -1, _trunc(shift), ss, flagMask(pe),
                     _trunc(filteredFlag), pe == "midpoint", opts=opts, out=out)
    if out is not None:
        return _pairs(out) if ss else out                                            # (R,) or the (2, R) view
    return pu[0]                                                                      # R/wrappers.R:118


def _tlen(tf, pe):
    """The tlenFilter() helper of R/wrappers.R:84-98 (named differently: `tlenFilter` is also an argument name)."""
    if pe == "ignore":
        return None
    if tf is None:
        return (0, 1000)
    if len(tf) != 2 or tf[0] < 0 or tf[1] < 0:
        raise ValueError("tlenFilter must be NULL or vector of 2 positive integers")
    if tf[0] > tf[1]:
        raise ValueError("tlenFilter[1] must be smaller or equal to tlenFilter[2]")
    return (int(tf[0]), int(tf[1]))


# runs=True: the profile as a ProfileRuns (run-length pairs per region and strand row) instead of a CountSignals; with
# device= its arrays are torch tensors on that device.
def bamProfile(bampath, gr, binsize=1, mapqual=0, shift=0, ss=False, paired_end=("ignore", "filter", "midpoint"),
               tlenFilter=None, filteredFlag=-1, verbose=False, opts=None, device=None, runs=False):
    if binsize < 1:
        raise ValueError("provide a binsize greater or equal to 1")                  # R/wrappers.R:136-137
    if binsize > 1 and isinstance(gr, GRanges) and (gr.width % int(binsize) != 0).any():
        warnings.warn("some ranges' widths are not a multiple of the selected binsize, "
                      "some bins will correspond to less than binsize basepairs")     # R/wrappers.R:138-141
    pe = _match_arg(paired_end, ("ignore", "filter", "midpoint"))
    bampath = os.path.expanduser(bampath)
    if runs:
        return profile_runs_core(bampath, gr, _tlen(tlenFilter, pe), _trunc(mapqual), _trunc(binsize), _trunc(shift), ss,
                                 flagMask(pe), _trunc(filteredFlag), pe == "midpoint", opts=opts, device=device)
    out = None if device is None else _empty_on(device, gr, _trunc(binsize), ss)
    flat, off = pileup_core(bampath, gr, _tlen(tlenFilter, pe), _trunc(mapqual), _trunc(binsize), _trunc(shift), ss,
                            flagMask(pe), _trunc(filteredFlag), pe == "midpoint", opts=opts, _lazy=True, out=out)
    return CountSignals(None, ss, flat=flat, offsets=off)


# runs=True: the coverage as a CoverageRuns (run-length pairs per region) instead of a CountSignals; with device= its
# arrays are torch tensors on that device.
# ss=True (beyond the R interface): strand-specific coverage, a (2, w) [sense; antisense] matrix per region.  A read's
# strand is its flag bit 0x10, relative to the region as in bamProfile; with paired_end="extend" only first mates count
# and a fragment goes to its first mate's strand.
def bamCoverage(bampath, gr, mapqual=0, paired_end=("ignore", "extend"), tlenFilter=None, filteredFlag=-1,
                verbose=False, opts=None, device=None, runs=False, ss=False):
    pe = _match_arg(paired_end, ("ignore", "extend"))
    bampath = os.path.expanduser(bampath)
    ss = bool(ss)
    if runs:
        return coverage_runs_core(bampath, gr, _tlen(tlenFilter, pe), _trunc(mapqual), flagMask(pe), _trunc(filteredFlag),
                                  pe == "extend", opts=opts, device=device, ss=ss)
    out = None if device is None else _empty_on(device, gr, 1, ss)
    flat, off = coverage_core(bampath, gr, _tlen(tlenFilter, pe), _trunc(mapqual), flagMask(pe), _trunc(filteredFlag),
                              pe == "extend", opts=opts, _lazy=True, out=out, ss=ss)
    return CountSignals(None, ss, flat=flat, offsets=off)
