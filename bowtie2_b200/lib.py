"""ctypes binding of libbt2g.so (C ABI: include/bt2g.h).

Names and argument meaning follow the reference calls each entry point replaces
(SeedAligner::exactSweep / searchAllSeeds, Ebwt::getOffset + joinedToTextOff, ...); see the
header for file:line citations.  All arrays are numpy; offsets travel as uint64.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

OFFMASK = np.uint64(0xFFFFFFFFFFFFFFFF)


class Bt2GpuError(RuntimeError):
    pass


def library_path() -> str:
    return os.path.join(_HERE, "libbt2g.so")


class _IndexHost(C.Structure):
    _fields_ = [
        ("off_size", C.c_int32), ("line_rate", C.c_int32), ("off_rate", C.c_int32), ("ftab_chars", C.c_int32),
        ("len", C.c_uint64), ("n_pat", C.c_uint64), ("n_frag", C.c_uint64),
        ("z_off_fw", C.c_uint64), ("z_off_bw", C.c_uint64), ("fchr", C.c_uint64 * 5),
        ("plen", C.c_void_p), ("rstarts", C.c_void_p), ("ebwt_fw", C.c_void_p), ("ebwt_bw", C.c_void_p),
        ("ftab_fw", C.c_void_p), ("eftab_fw", C.c_void_p), ("ftab_bw", C.c_void_p), ("eftab_bw", C.c_void_p),
        ("offs", C.c_void_p), ("n_recs", C.c_uint64), ("rec_off", C.c_void_p), ("rec_len", C.c_void_p),
        ("rec_first", C.c_void_p), ("ref_buf", C.c_void_p),
    ]


class _IndexInfo(C.Structure):
    _fields_ = [
        ("off_size", C.c_int32), ("line_rate", C.c_int32), ("off_rate", C.c_int32), ("ftab_chars", C.c_int32),
        ("len", C.c_uint64), ("bwt_len", C.c_uint64), ("num_sides", C.c_uint64), ("side_sz", C.c_uint64),
        ("side_bwt_sz", C.c_uint64), ("side_bwt_len", C.c_uint64), ("ebwt_tot_len", C.c_uint64),
        ("offs_len", C.c_uint64), ("ftab_len", C.c_uint64), ("eftab_len", C.c_uint64), ("n_pat", C.c_uint64),
        ("n_frag", C.c_uint64), ("n_recs", C.c_uint64), ("ref_buf_bytes", C.c_uint64),
        ("z_off_fw", C.c_uint64), ("z_off_bw", C.c_uint64), ("fchr", C.c_uint64 * 5),
        ("has_bw", C.c_int32), ("has_ref", C.c_int32), ("device_bytes", C.c_uint64),
    ]


class _Reads(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("seq", C.c_void_p), ("qual", C.c_void_p), ("off", C.c_void_p)]


class _SeedPlan(C.Structure):
    _fields_ = [("seed_len", C.c_int32), ("max_seeds", C.c_int32), ("nofw", C.c_int32), ("norc", C.c_int32),
                ("interval", C.c_void_p), ("offset", C.c_void_p)]


# every symbol include/bt2g.h declares; tests assert the built library exports all of them
EXPORTS = [
    "bt2g_create", "bt2g_destroy", "bt2g_last_error", "bt2g_abi_version",
    "bt2g_load_index_files", "bt2g_load_index_host", "bt2g_load_index_device",
    "bt2g_index_info_get", "bt2g_index_array",
    "bt2g_rank4", "bt2g_maplf1", "bt2g_maplf_range", "bt2g_ftab_lohi",
    "bt2g_exact_sweep", "bt2g_seed_search", "bt2g_resolve", "bt2g_get_stretch",
]


def load_library() -> C.CDLL:
    """Load libbt2g.so; raise (never fall back) when it has not been built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise Bt2GpuError(f"{path} not built: run `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(path)
    vp, u64, i32 = C.c_void_p, C.c_uint64, C.c_int
    lib.bt2g_create.argtypes = [i32, C.POINTER(vp)]
    lib.bt2g_destroy.argtypes = [vp]
    lib.bt2g_destroy.restype = None
    lib.bt2g_last_error.argtypes = [vp]
    lib.bt2g_last_error.restype = C.c_char_p
    lib.bt2g_load_index_files.argtypes = [vp, C.c_char_p]
    lib.bt2g_load_index_files_ex.argtypes = [vp, C.c_char_p, i32]
    lib.bt2g_load_index_host.argtypes = [vp, C.POINTER(_IndexHost)]
    lib.bt2g_load_index_device.argtypes = [vp, C.POINTER(_IndexHost)]
    lib.bt2g_index_info_get.argtypes = [vp, C.POINTER(_IndexInfo)]
    lib.bt2g_index_array.argtypes = [vp, i32, C.POINTER(vp), C.POINTER(u64)]
    lib.bt2g_rank4.argtypes = [vp, i32, vp, u64, vp]
    lib.bt2g_maplf1.argtypes = [vp, i32, vp, vp, u64, vp]
    lib.bt2g_maplf_range.argtypes = [vp, i32, vp, vp, u64, vp, vp, vp]
    lib.bt2g_ftab_lohi.argtypes = [vp, i32, vp, u64, vp]
    lib.bt2g_exact_sweep.argtypes = [vp, C.POINTER(_Reads), i32, i32, vp, vp]
    lib.bt2g_seed_search.argtypes = [vp, C.POINTER(_Reads), C.POINTER(_SeedPlan), vp, vp]
    lib.bt2g_resolve.argtypes = [vp, vp, vp, u64, i32, vp, vp, vp, vp, vp]
    lib.bt2g_get_stretch.argtypes = [vp, vp, vp, vp, u64, C.c_int32, vp]
    _LIB = lib
    return lib


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _c(a, dtype) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=dtype)


class ReadBatch:
    """Reads as the hot path sees them: codes 0..3 = ACGT, 4 = N; Phred+33 qualities."""

    def __init__(self, seq: np.ndarray, off: np.ndarray, qual: Optional[np.ndarray] = None):
        self.seq = _c(seq, np.uint8)
        self.off = _c(off, np.uint64)
        self.qual = None if qual is None else _c(qual, np.uint8)
        self.n = len(self.off) - 1

    @classmethod
    def from_list(cls, reads, quals=None):
        lens = np.array([len(r) for r in reads], dtype=np.uint64)
        off = np.zeros(len(reads) + 1, dtype=np.uint64)
        np.cumsum(lens, out=off[1:])
        seq = np.concatenate([np.asarray(r, dtype=np.uint8) for r in reads]) if len(reads) else np.zeros(0, np.uint8)
        q = None
        if quals is not None:
            q = np.concatenate([np.asarray(x, dtype=np.uint8) for x in quals]) if len(quals) else np.zeros(0, np.uint8)
        return cls(seq, off, q)

    def lengths(self) -> np.ndarray:
        return (self.off[1:] - self.off[:-1]).astype(np.int64)

    def _struct(self) -> _Reads:
        return _Reads(self.n, _ptr(self.seq), _ptr(self.qual), _ptr(self.off))


class Bt2Gpu:
    """One context per GPU (include/bt2g.h).  Raises Bt2GpuError on any failure."""

    def __init__(self, device: int = 0):
        self._lib = load_library()
        h = C.c_void_p()
        rc = self._lib.bt2g_create(device, C.byref(h))
        if rc != 0:
            raise Bt2GpuError(f"bt2g_create(device={device}) failed with {rc}: no usable CUDA device")
        self._h = h
        self.device = device
        self._keep = []

    def close(self):
        if getattr(self, "_h", None):
            self._lib.bt2g_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str):
        if rc != 0:
            msg = self._lib.bt2g_last_error(self._h)
            raise Bt2GpuError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")

    # ---- index ---------------------------------------------------------------------
    def load_index_files(self, basename: str, offrate: int = -1):
        """offrate > the index's own offRate keeps every 2^diff-th SA sample (bowtie2 --offrate, bt2_io.cpp:217-230)."""
        if offrate >= 0:
            self._check(self._lib.bt2g_load_index_files_ex(self._h, basename.encode(), int(offrate)), "bt2g_load_index_files_ex")
        else:
            self._check(self._lib.bt2g_load_index_files(self._h, basename.encode()), "bt2g_load_index_files")

    def load_index_host(self, index_file: "IndexFile"):
        """Upload a host image read with IndexFile (bt2g_load_index_host copies; the image may be closed afterwards)."""
        self._check(self._lib.bt2g_load_index_host(self._h, C.byref(index_file.desc)), "bt2g_load_index_host")

    def load_index_device(self, desc: dict, keep=None):
        """Adopt device arrays (e.g. torch tensors filled by an NCCL broadcast). `desc` maps
        bt2g_index_host field names to ints (scalars / raw device pointers)."""
        ih = _IndexHost()
        for k, v in desc.items():
            if k == "fchr":
                for i in range(5):
                    ih.fchr[i] = int(v[i])
            else:
                setattr(ih, k, v)
        self._keep = keep
        self._check(self._lib.bt2g_load_index_device(self._h, C.byref(ih)), "bt2g_load_index_device")

    def info(self) -> dict:
        inf = _IndexInfo()
        self._check(self._lib.bt2g_index_info_get(self._h, C.byref(inf)), "bt2g_index_info_get")
        d = {k: getattr(inf, k) for k, _ in _IndexInfo._fields_ if k != "fchr"}
        d["fchr"] = [int(x) for x in inf.fchr]
        return d

    def index_array(self, which: int):
        p, b = C.c_void_p(), C.c_uint64()
        self._check(self._lib.bt2g_index_array(self._h, which, C.byref(p), C.byref(b)), "bt2g_index_array")
        return (p.value or 0), int(b.value)

    # ---- FM primitives -------------------------------------------------------------
    def rank4(self, rows, mirror: bool = False) -> np.ndarray:
        rows = _c(rows, np.uint64)
        out = np.empty((len(rows), 4), dtype=np.uint64)
        self._check(self._lib.bt2g_rank4(self._h, int(mirror), _ptr(rows), len(rows), _ptr(out)), "bt2g_rank4")
        return out

    def maplf1(self, rows, chars, mirror: bool = False) -> np.ndarray:
        rows, chars = _c(rows, np.uint64), _c(chars, np.uint8)
        out = np.empty(len(rows), dtype=np.uint64)
        self._check(self._lib.bt2g_maplf1(self._h, int(mirror), _ptr(rows), _ptr(chars), len(rows), _ptr(out)), "bt2g_maplf1")
        return out

    def maplf_range(self, tops, nums, mirror: bool = False):
        """Ebwt::mapLFRange (bt2_idx.h:2268) for every [top, top+num): (upto[n,4], in[n,4], chars: one BWT character per
        row, the ranges back to back)."""
        tops, nums = _c(tops, np.uint64), _c(nums, np.uint64)
        upto = np.empty((len(tops), 4), dtype=np.uint64)
        inn = np.empty((len(tops), 4), dtype=np.uint64)
        chars = np.empty(int(nums.sum()), dtype=np.uint8)
        self._check(self._lib.bt2g_maplf_range(self._h, int(mirror), _ptr(tops), _ptr(nums), len(tops), _ptr(upto), _ptr(inn), _ptr(chars)),
                    "bt2g_maplf_range")
        return upto, inn, chars

    def ftab_lohi(self, idx, mirror: bool = False) -> np.ndarray:
        idx = _c(idx, np.uint64)
        out = np.empty((len(idx), 2), dtype=np.uint64)
        self._check(self._lib.bt2g_ftab_lohi(self._h, int(mirror), _ptr(idx), len(idx), _ptr(out)), "bt2g_ftab_lohi")
        return out

    # ---- K1 ------------------------------------------------------------------------
    def exact_sweep(self, reads: ReadBatch, nofw=False, norc=False):
        mine = np.empty((reads.n, 2), dtype=np.uint8)
        ee = np.empty((reads.n, 4), dtype=np.uint64)
        st = reads._struct()
        self._check(self._lib.bt2g_exact_sweep(self._h, C.byref(st), int(nofw), int(norc), _ptr(mine), _ptr(ee)), "bt2g_exact_sweep")
        return mine, ee

    def seed_search(self, reads: ReadBatch, seed_len: int, interval, offset, max_seeds: int, nofw=False, norc=False):
        interval = _c(np.broadcast_to(interval, (reads.n,)), np.int32)
        offset = _c(np.broadcast_to(offset, (reads.n,)), np.int32)
        out = np.empty((reads.n, 2, max_seeds, 4), dtype=np.uint64)
        ns = np.empty(reads.n, dtype=np.int32)
        plan = _SeedPlan(seed_len, max_seeds, int(nofw), int(norc), _ptr(interval), _ptr(offset))
        st = reads._struct()
        self._check(self._lib.bt2g_seed_search(self._h, C.byref(st), C.byref(plan), _ptr(out), _ptr(ns)), "bt2g_seed_search")
        return out, ns

    # ---- K2 ------------------------------------------------------------------------
    def resolve(self, rows, hitlen, reject_straddle=False):
        rows = _c(rows, np.uint64)
        n = len(rows)
        hitlen = _c(np.broadcast_to(hitlen, (n,)), np.uint32)
        joined, tidx, textoff, tlen = (np.empty(n, dtype=np.uint64) for _ in range(4))
        flags = np.empty(n, dtype=np.uint8)
        self._check(self._lib.bt2g_resolve(self._h, _ptr(rows), _ptr(hitlen), n, int(reject_straddle), _ptr(joined),
                                           _ptr(tidx), _ptr(textoff), _ptr(tlen), _ptr(flags)), "bt2g_resolve")
        return joined, tidx, textoff, tlen, flags

    def get_stretch(self, tidx, off, count, stride: int) -> np.ndarray:
        tidx, off, count = _c(tidx, np.uint64), _c(off, np.int64), _c(count, np.int32)
        out = np.empty((len(tidx), stride), dtype=np.uint8)
        self._check(self._lib.bt2g_get_stretch(self._h, _ptr(tidx), _ptr(off), _ptr(count), len(tidx), stride, _ptr(out)), "bt2g_get_stretch")
        return out


# ---- K3: extension DP -----------------------------------------------------------------------
class _Scoring(C.Structure):
    _fields_ = [("match_bonus", C.c_int32), ("rdgap_const", C.c_int32), ("rdgap_linear", C.c_int32),
                ("rfgap_const", C.c_int32), ("rfgap_linear", C.c_int32), ("gapbar", C.c_int32),
                ("local", C.c_int32), ("mmpen", C.c_uint8 * 64), ("npen", C.c_uint8 * 64),
                ("nceil_const", C.c_double), ("nceil_linear", C.c_double)]      # = bt2g_scoring (include/bt2g.h), 176 bytes


DP_PROBLEM = np.dtype([("read_idx", "<u4"), ("fw", "<u4"), ("tidx", "<u8"), ("refl", "<i8"), ("refr", "<i8"),
                       ("triml", "<i4"), ("corel", "<i4"), ("corer", "<i4"), ("minsc", "<i4"),
                       ("nceil", "<i4"), ("reserved", "<i4")], align=True)
DP_SUMMARY = np.dtype([("found", "<i4"), ("best", "<i4"), ("ncand", "<i4"), ("naln", "<i4"), ("flags", "<i4")])
DP_CAND = np.dtype([("score", "<i4"), ("row", "<i4"), ("col", "<i4"), ("fate", "<i4")])
DP_ALN = np.dtype([("cand_idx", "<i4"), ("score", "<i4"), ("ns", "<i4"), ("gaps", "<i4"), ("refns", "<i4"),
                   ("row0", "<i4"), ("col0", "<i4"), ("trim_beg", "<i4"), ("trim_end", "<i4"), ("nops", "<i4")])

EXPORTS += ["bt2g_scoring_default", "bt2g_set_scoring", "bt2g_set_dp_mode", "bt2g_set_extend_mode", "bt2g_dp_extend"]

OP_MATCH, OP_MM, OP_REFGAP, OP_READGAP = 0, 1, 2, 3
EDIT_READ_GAP, EDIT_REF_GAP, EDIT_MM = 1, 2, 3      # edit.h:34-39


def _bind_dp(lib):
    if getattr(lib, "_dp_bound", False):
        return
    vp = C.c_void_p
    lib.bt2g_scoring_default.argtypes = [C.POINTER(_Scoring), C.c_int]
    lib.bt2g_scoring_default.restype = None
    lib.bt2g_set_scoring.argtypes = [vp, C.POINTER(_Scoring)]
    lib.bt2g_dp_extend.argtypes = [vp, C.POINTER(_Reads), vp, C.c_uint64, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, vp]
    lib._dp_bound = True


def _set_scoring(self, local: bool = False, **over):
    """Install the scoring scheme (reference defaults, scoring.h:28-84; override by keyword)."""
    _bind_dp(self._lib)
    sc = _Scoring()
    self._lib.bt2g_scoring_default(C.byref(sc), int(local))
    for k, v in over.items():
        setattr(sc, k, v)
    self._check(self._lib.bt2g_set_scoring(self._h, C.byref(sc)), "bt2g_set_scoring")
    self.scoring = sc


def _set_scoring_policy(self, sc, local: bool = None):
    """Install the device scoring that corresponds to a policy.Scoring (--ma / --mp / --np / --rdg / --rfg / --n-ceil): the
    same object the exact policy derives minsc / perfect / MAPQ from, so kernels and policy cannot disagree."""
    from . import policy
    local = bool(sc.local if local is None else local)
    nce = sc.n_ceil_func()
    mm = (C.c_uint8 * 64)(*[policy.mm_penalty(min(q, 40), sc.mmp_max, sc.mmp_min) for q in range(64)])
    np_ = (C.c_uint8 * 64)(*[sc.n_pen] * 64)
    self.set_scoring(local=local, match_bonus=sc.match_bonus, rdgap_const=sc.rdgap_const, rdgap_linear=sc.rdgap_linear,
                     rfgap_const=sc.rfgap_const, rfgap_linear=sc.rfgap_linear, gapbar=sc.gapbar, mmpen=mm, npen=np_,
                     nceil_const=float(nce.C), nceil_linear=float(nce.L))


def _set_dp_mode(self, cap: int):
    """bt2g_set_dp_mode: cap the end-to-end DP kernel generation of this context: 0, 1 or 3 (the default); 2 acts as 1"""
    self._lib.bt2g_set_dp_mode.argtypes = [C.c_void_p, C.c_int]
    self._check(self._lib.bt2g_set_dp_mode(self._h, int(cap)), "bt2g_set_dp_mode")


def _dp_extend(self, reads: ReadBatch, probs: np.ndarray, max_cands=128, max_alns=4, max_ops=None):
    """SwAligner::initRef + align + nextAlignment* for each problem (include/bt2g.h)."""
    _bind_dp(self._lib)
    assert probs.dtype == DP_PROBLEM
    probs = np.ascontiguousarray(probs)
    n = len(probs)
    if max_ops is None:
        max_ops = int(reads.lengths().max()) + 64 if reads.n else 64
    summ = np.zeros(n, dtype=DP_SUMMARY)
    cands = np.zeros((n, max_cands), dtype=DP_CAND)
    alns = np.zeros((n, max_alns), dtype=DP_ALN)
    ops = np.zeros((n, max_alns, max_ops), dtype=np.uint8)
    st = reads._struct()
    self._check(self._lib.bt2g_dp_extend(self._h, C.byref(st), _ptr(probs), n, max_cands, max_alns, max_ops,
                                         _ptr(summ), _ptr(cands), _ptr(alns), _ptr(ops)), "bt2g_dp_extend")
    return summ, cands, alns, ops


Bt2Gpu.set_scoring = _set_scoring
Bt2Gpu.set_scoring_policy = _set_scoring_policy
def _set_extend_mode(self, through_text: bool):
    """bt2g_set_extend_mode: unique seed hits extended against the packed reference (default) or by walking the index"""
    self._lib.bt2g_set_extend_mode.argtypes = [C.c_void_p, C.c_int]
    self._check(self._lib.bt2g_set_extend_mode(self._h, int(bool(through_text))), "bt2g_set_extend_mode")


Bt2Gpu.set_dp_mode = _set_dp_mode
Bt2Gpu.set_extend_mode = _set_extend_mode
Bt2Gpu.dp_extend = _dp_extend


def ops_to_edits(ops: np.ndarray, nops: int, read_codes: np.ndarray, fw: bool, row0: int, trim_end: int = 0):
    """Rebuild the reference's Edit list (edit.h:57-) from a device op string.

    The device lists columns from the last read row back to the first; the reference builds
    `ned` in the same order and reverses it (SwResult::reverse), then inverts positions for
    reverse-complement alignments (AlnRes::invertEdits via nextAlignment, aligner_sw.cpp:1135).
    Returns a list of (pos, chr, qchr, type) with chr/qchr as ASCII codes, pos w.r.t. the 5'
    end of the original read -- the representation SAM printing consumes."""
    dna = b"ACGTN"
    rdlen = len(read_codes)
    seq = read_codes if fw else np.array([4 if c > 3 else 3 - c for c in read_codes[::-1]], dtype=np.uint8)
    fwd = ops[:nops][::-1]
    row = row0
    out = []
    for op in fwd:
        typ, refc = int(op) & 3, (int(op) >> 2) & 7
        if typ == OP_MATCH:
            row += 1
        elif typ == OP_MM:
            out.append([row - row0, dna[refc], dna[seq[row]], EDIT_MM])
            row += 1
        elif typ == OP_REFGAP:
            out.append([row - row0, ord("-"), dna[seq[row]], EDIT_REF_GAP])
            row += 1
        else:
            out.append([row - row0, dna[refc], ord("-"), EDIT_READ_GAP])
    if not fw:
        # AlnRes::invertEdits -> Edit::invertPoss (edit.cpp:50-78)
        # positions are relative to the soft-trimmed extent (AlnRes::setShape, aligner_result.cpp:101-117)
        ext = rdlen - row0 - trim_end
        out = out[::-1]
        for e in out:
            e[0] = ext - e[0] - (0 if e[3] == EDIT_READ_GAP else 1)
    return out


# ---- batched hot path ------------------------------------------------------------------------
class _PipeParams(C.Structure):
    _fields_ = [("seed_len", C.c_int32), ("max_seeds", C.c_int32), ("row_cap", C.c_int32), ("range_max", C.c_int32),
                ("max_len", C.c_int32), ("maxhalf", C.c_int32), ("max_cands", C.c_int32), ("max_alns", C.c_int32),
                ("max_ops", C.c_int32), ("max_probs", C.c_int32), ("minsc_by_len", C.c_void_p), ("nceil_by_len", C.c_void_p),
                ("nceil_raw_by_len", C.c_void_p), ("interval_by_len", C.c_void_p), ("rdgaps_by_len", C.c_void_p),
                ("rfgaps_by_len", C.c_void_p)]


READ_RESULT = np.dtype([("found", "<i4"), ("score", "<i4"), ("score2", "<i4"), ("fw", "<u4"), ("tidx", "<u8"),
                        ("refoff", "<i8"), ("nops", "<i4"), ("ndp", "<i4"), ("trim_left", "<i4"), ("trim_right", "<i4"),
                        ("mapq", "<i4"), ("pad", "<i4")], align=True)

EXPORTS += ["bt2g_pipeline_create", "bt2g_pipeline_destroy", "bt2g_pipeline_run_dev", "bt2g_pipeline_run_host",
            "bt2g_pipeline_results_dev", "bt2g_pipeline_counters", "bt2g_pipeline_stage_ms", "bt2g_pipeline_kernel_launches",
            "bt2g_pipeline_enable_pairs", "bt2g_pipeline_run_paired_dev", "bt2g_pipeline_run_paired_host",
            "bt2g_pipeline_pairs_dev", "bt2g_pipeline_pair_counters", "bt2g_pipeline_pair_stage_ms"]
PAIR_RESULT = np.dtype([("pair_type", "<i4"), ("kind", "<i4"), ("source", "<i4"), ("score_sum", "<i4"), ("fraglen", "<i8")], align=True)


class Pipeline:
    """bt2g_pipeline: the batched hot path for one preset / scoring scheme (include/bt2g.h)."""

    def __init__(self, gpu: "Bt2Gpu", preset_name: str = "sensitive", max_len: int = 100, max_reads: int = 1 << 20,
                 row_cap: int = 16, range_max: int = 8, max_cands: int = 64, max_alns: int = 2, local: bool = False,
                 both_mates: bool = False, max_probs: int = 0):
        from . import policy
        self.gpu = gpu
        lib = gpu._lib
        _bind_dp(lib)
        vp = C.c_void_p
        lib.bt2g_pipeline_create.argtypes = [vp, C.POINTER(_PipeParams), C.c_uint64, C.c_uint64, C.POINTER(vp)]
        lib.bt2g_pipeline_destroy.argtypes = [vp]
        lib.bt2g_pipeline_destroy.restype = None
        lib.bt2g_pipeline_run_dev.argtypes = [vp, vp, vp, vp, C.c_uint64, vp, C.c_int]
        lib.bt2g_pipeline_run_host.argtypes = [vp, C.POINTER(_Reads), vp, vp]
        lib.bt2g_pipeline_results_dev.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
        lib.bt2g_pipeline_counters.argtypes = [vp, vp]
        lib.bt2g_pipeline_stage_ms.argtypes = [vp, vp]
        gpu.set_scoring(local=local)
        sc = policy.Scoring.default(local)
        pre = policy.preset(preset_name, local)
        L1 = max_len + 1
        lens = np.arange(L1)
        tab = lambda f: np.array([f(int(x)) if x > 0 else 0 for x in lens], dtype=np.int32)
        self._tabs = [tab(sc.min_score), tab(sc.n_ceil), tab(sc.n_ceil_raw),
                      tab(lambda x: policy.seed_interval(pre.ival, x, both_mates)),
                      tab(lambda x: sc.max_read_gaps(sc.min_score(x), x)), tab(lambda x: sc.max_ref_gaps(sc.min_score(x), x))]
        self.max_ops = max_len + 64
        self.seed_len = pre.seed_len
        # seeds per strand the buffers must hold: the largest count any read length up to max_len produces with ITS
        # OWN interval (the smallest interval belongs to the shortest reads, which have the fewest positions)
        self.max_seeds = max(1, max(policy.n_seeds(l, pre.seed_len, max(int(self._tabs[3][l]), 1)) for l in range(1, L1)))
        prm = _PipeParams(pre.seed_len, self.max_seeds, row_cap, range_max, max_len, 15, max_cands, max_alns, self.max_ops, max_probs,
                          *[_ptr(t) for t in self._tabs])
        h = vp()
        gpu._check(lib.bt2g_pipeline_create(gpu._h, C.byref(prm), max_reads, max_reads * max_len, C.byref(h)), "bt2g_pipeline_create")
        self._h = h
        self.max_reads, self.max_len = max_reads, max_len

    def close(self):
        if getattr(self, "_h", None):
            self.gpu._lib.bt2g_pipeline_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- paired-end pass (include/bt2g.h: bt2g_pipeline_enable_pairs ...) ----
    def enable_pairs(self, pe=None):
        from . import policy
        lib = self.gpu._lib
        vp = C.c_void_p
        lib.bt2g_pipeline_enable_pairs.argtypes = [vp, vp]
        lib.bt2g_pipeline_run_paired_dev.argtypes = [vp, vp, vp, vp, C.c_uint64, vp, C.c_int]
        lib.bt2g_pipeline_run_paired_host.argtypes = [vp, C.POINTER(_Reads), vp, vp, vp]
        lib.bt2g_pipeline_pairs_dev.argtypes = [vp, C.POINTER(vp)]
        lib.bt2g_pipeline_pair_counters.argtypes = [vp, vp]
        lib.bt2g_pipeline_pair_stage_ms.argtypes = [vp, vp]
        self.pe = pe if pe is not None else policy.PairedEndPolicy()
        pp = _pe_struct(self.pe)
        self.gpu._check(lib.bt2g_pipeline_enable_pairs(self._h, C.byref(pp)), "bt2g_pipeline_enable_pairs")

    def run_paired_host(self, reads: ReadBatch, want_ops: bool = True):
        """reads: mate 1 / mate 2 interleaved -> (per-read results, ops, per-pair results)."""
        res = np.zeros(reads.n, dtype=READ_RESULT)
        ops = np.zeros((reads.n, self.max_ops), dtype=np.uint8) if want_ops else None
        pairs = np.zeros(reads.n // 2, dtype=PAIR_RESULT)
        st = reads._struct()
        self.gpu._check(self.gpu._lib.bt2g_pipeline_run_paired_host(self._h, C.byref(st), _ptr(res), _ptr(ops), _ptr(pairs)),
                        "bt2g_pipeline_run_paired_host")
        return res, ops, pairs

    def run_paired_dev(self, d_seq: int, d_qual: int, d_off: int, n_pairs: int, stream: int = 0, count: bool = False):
        self.gpu._check(self.gpu._lib.bt2g_pipeline_run_paired_dev(self._h, d_seq, d_qual, d_off, n_pairs, stream, int(count)),
                        "bt2g_pipeline_run_paired_dev")

    def pair_counters(self) -> dict:
        out = np.zeros(2, dtype=np.uint64)
        self.gpu._check(self.gpu._lib.bt2g_pipeline_pair_counters(self._h, _ptr(out)), "bt2g_pipeline_pair_counters")
        return {"mate_problems": int(out[0]), "mate_cells": int(out[1])}

    def pair_stage_ms(self) -> dict:
        out = np.zeros(3, dtype=np.float32)
        self.gpu._check(self.gpu._lib.bt2g_pipeline_pair_stage_ms(self._h, _ptr(out)), "bt2g_pipeline_pair_stage_ms")
        return dict(zip(("frame_mates", "mate_dp", "pick_pairs"), (float(x) for x in out)))

    def kernel_launches(self) -> int:
        self.gpu._lib.bt2g_pipeline_kernel_launches.argtypes = [C.c_void_p]
        return int(self.gpu._lib.bt2g_pipeline_kernel_launches(self._h))

    def run_host(self, reads: ReadBatch, want_ops: bool = True):
        res = np.zeros(reads.n, dtype=READ_RESULT)
        ops = np.zeros((reads.n, self.max_ops), dtype=np.uint8) if want_ops else None
        st = reads._struct()
        self.gpu._check(self.gpu._lib.bt2g_pipeline_run_host(self._h, C.byref(st), _ptr(res), _ptr(ops)), "bt2g_pipeline_run_host")
        return res, ops

    def run_dev(self, d_seq: int, d_qual: int, d_off: int, n_reads: int, stream: int = 0, count: bool = False):
        self.gpu._check(self.gpu._lib.bt2g_pipeline_run_dev(self._h, d_seq, d_qual, d_off, n_reads, stream or None, int(count)),
                        "bt2g_pipeline_run_dev")

    def counters(self) -> dict:
        out = np.zeros(6, dtype=np.uint64)
        self.gpu._check(self.gpu._lib.bt2g_pipeline_counters(self._h, _ptr(out)), "bt2g_pipeline_counters")
        k = ["sweep_sides", "seed_sides", "resolve_sides", "dp_cells", "dp_problems", "reads"]
        return {a: int(b) for a, b in zip(k, out)}

    STAGES = ["plan", "exact_sweep", "seed_search", "collect", "resolve", "frame", "dp", "pick"]

    def stage_ms(self) -> dict:
        out = np.zeros(8, dtype=np.float32)
        self.gpu._check(self.gpu._lib.bt2g_pipeline_stage_ms(self._h, _ptr(out)), "bt2g_pipeline_stage_ms")
        return {k: float(v) for k, v in zip(self.STAGES, out)}

    def results_dev(self):
        r, o = C.c_void_p(), C.c_void_p()
        self.gpu._check(self.gpu._lib.bt2g_pipeline_results_dev(self._h, C.byref(r), C.byref(o)), "bt2g_pipeline_results_dev")
        return r.value, o.value


def ops_to_cigar(ops: np.ndarray, nops: int, trim_left: int = 0, trim_right: int = 0) -> str:
    """SAM CIGAR of a device op string (reference: AlnRes::printCigar via StackedAln,
    aligner_result.cpp): M for match/mismatch, I for a reference gap, D for a read gap, S for
    the soft-trimmed ends of a local alignment."""
    sym = {OP_MATCH: "M", OP_MM: "M", OP_REFGAP: "I", OP_READGAP: "D"}
    out, run, last = [], 0, None
    if trim_left:
        out.append(f"{trim_left}S")
    for op in ops[:nops][::-1]:
        s = sym[int(op) & 3]
        if s == last:
            run += 1
        else:
            if last is not None:
                out.append(f"{run}{last}")
            last, run = s, 1
    if last is not None:
        out.append(f"{run}{last}")
    if trim_right:
        out.append(f"{trim_right}S")
    return "".join(out)


# ---- SwDriver::extend ------------------------------------------------------------------------
EXPORTS += ["bt2g_extend_exact"]


def _extend_exact(self, reads: ReadBatch, seed_len: int, interval, offset, max_seeds: int, ranges: np.ndarray) -> np.ndarray:
    """nlex/nrex of every seed hit (include/bt2g.h: bt2g_extend_exact) -> uint8 [n, 2, max_seeds, 2]."""
    lib = self._lib
    lib.bt2g_extend_exact.argtypes = [C.c_void_p, C.POINTER(_Reads), C.POINTER(_SeedPlan), C.c_void_p, C.c_void_p]
    interval = _c(np.broadcast_to(interval, (reads.n,)), np.int32)
    offset = _c(np.broadcast_to(offset, (reads.n,)), np.int32)
    ranges = _c(ranges, np.uint64)
    out = np.zeros((reads.n, 2, max_seeds, 2), dtype=np.uint8)
    plan = _SeedPlan(seed_len, max_seeds, 0, 0, _ptr(interval), _ptr(offset))
    st = reads._struct()
    self._check(lib.bt2g_extend_exact(self._h, C.byref(st), C.byref(plan), _ptr(ranges), _ptr(out)), "bt2g_extend_exact")
    return out


Bt2Gpu.extend_exact = _extend_exact


# ---- SeedAligner::oneMmSearch ------------------------------------------------------------------
EXPORTS += ["bt2g_one_mm"]
MM_HIT = np.dtype([("top", "<u8"), ("bot", "<u8"), ("pos", "<i4"), ("chr", "<i4"), ("qchr", "<i4"), ("score", "<i4")])


def _one_mm(self, reads: ReadBatch, minsc, strand_mask=3, max_hits: int = 16):
    """1-mismatch end-to-end hits (include/bt2g.h: bt2g_one_mm) -> (hits [n,4,max_hits], counts [n,4])."""
    lib = self._lib
    lib.bt2g_one_mm.argtypes = [C.c_void_p, C.POINTER(_Reads), C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
    minsc = _c(np.broadcast_to(minsc, (reads.n,)), np.int32)
    mask = _c(np.broadcast_to(strand_mask, (reads.n,)), np.uint8)
    hits = np.zeros((reads.n, 4, max_hits), dtype=MM_HIT)
    counts = np.zeros((reads.n, 4), dtype=np.int32)
    st = reads._struct()
    self._check(lib.bt2g_one_mm(self._h, C.byref(st), _ptr(minsc), _ptr(mask), max_hits, _ptr(hits), _ptr(counts)), "bt2g_one_mm")
    return hits, counts


Bt2Gpu.one_mm = _one_mm


# ---- paired-end framing (PairedEndPolicy::otherMate + DynProgFramer::frameFindMateRect, peClassifyPair) ----
EXPORTS += ["bt2g_frame_mate", "bt2g_pe_classify"]
MATE_ANCHOR = np.dtype([("off", "<i8"), ("reflen", "<u8"), ("len1", "<u4"), ("len2", "<u4"), ("maxalcols", "<i4"),
                        ("maxrdgap", "<i4"), ("maxrfgap", "<i4"), ("maxns", "<i4"), ("maxhalf", "<i4"),
                        ("is1", "u1"), ("fw", "u1"), ("pad", "u1", (2,))], align=True)
MATE_FRAME = np.dtype([("status", "<i4"), ("oleft", "u1"), ("ofw", "u1"), ("pad", "u1", (2,)),
                       ("oll", "<i8"), ("olr", "<i8"), ("orl", "<i8"), ("orr", "<i8"),
                       ("refl", "<i8"), ("refr", "<i8"), ("refl_pretrim", "<i8"), ("refr_pretrim", "<i8"),
                       ("triml", "<i8"), ("trimr", "<i8"), ("corel", "<i8"), ("corer", "<i8"), ("maxgap", "<i8")], align=True)


class _PePolicy(C.Structure):
    _fields_ = [("pol", C.c_int32), ("flags", C.c_int32), ("maxfrag", C.c_uint64), ("minfrag", C.c_uint64)]


def _pe_struct(pe) -> _PePolicy:
    """policy.PairedEndPolicy -> bt2g_pe_policy (the local flag does not enter this arithmetic)."""
    return _PePolicy(int(pe.pol), int(pe.flags()) & 31, int(pe.maxfrag), int(pe.minfrag))


def _frame_mate(self, pe, anchors: np.ndarray) -> np.ndarray:
    """include/bt2g.h: bt2g_frame_mate.  anchors: MATE_ANCHOR array -> MATE_FRAME array."""
    lib = self._lib
    lib.bt2g_frame_mate.argtypes = [C.c_void_p, C.POINTER(_PePolicy), C.c_void_p, C.c_uint64, C.c_void_p]
    anchors = np.ascontiguousarray(anchors, dtype=MATE_ANCHOR)
    out = np.zeros(len(anchors), dtype=MATE_FRAME)
    pp = _pe_struct(pe)
    self._check(lib.bt2g_frame_mate(self._h, C.byref(pp), _ptr(anchors), len(anchors), _ptr(out)), "bt2g_frame_mate")
    return out


def _pe_classify(self, pe, pairs: np.ndarray) -> np.ndarray:
    """include/bt2g.h: bt2g_pe_classify.  pairs: int64 [n, 6] = off1, len1, fw1, off2, len2, fw2."""
    lib = self._lib
    lib.bt2g_pe_classify.argtypes = [C.c_void_p, C.POINTER(_PePolicy), C.c_void_p, C.c_uint64, C.c_void_p]
    pairs = np.ascontiguousarray(pairs, dtype=np.int64).reshape(-1, 6)
    out = np.zeros(len(pairs), dtype=np.int32)
    pp = _pe_struct(pe)
    self._check(lib.bt2g_pe_classify(self._h, C.byref(pp), _ptr(pairs), len(pairs), _ptr(out)), "bt2g_pe_classify")
    return out


Bt2Gpu.frame_mate = _frame_mate
Bt2Gpu.pe_classify = _pe_classify


# ---- SwAligner::ungappedAlign ---------------------------------------------------------------------
EXPORTS += ["bt2g_ungapped"]
UNGAPPED_PROBLEM = np.dtype([("read_idx", "<u4"), ("fw", "<u4"), ("tidx", "<u8"), ("refoff", "<i8"), ("reflen", "<u8"),
                             ("minsc", "<i4"), ("ohang", "<i4")], align=True)
UNGAPPED_RESULT = np.dtype([("status", "<i4"), ("score", "<i4"), ("rowi", "<i4"), ("rowf", "<i4"), ("ns", "<i4"),
                            ("refns", "<i4"), ("nedits", "<i4"), ("pad", "<i4")], align=True)


def _ungapped(self, reads: ReadBatch, probs: np.ndarray, want_mask: bool = True):
    """include/bt2g.h: bt2g_ungapped -> (results, edit mask [n, max_len] or None)."""
    lib = self._lib
    lib.bt2g_ungapped.argtypes = [C.c_void_p, C.POINTER(_Reads), C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint32]
    probs = np.ascontiguousarray(probs, dtype=UNGAPPED_PROBLEM)
    out = np.zeros(len(probs), dtype=UNGAPPED_RESULT)
    stride = int(reads.lengths().max()) if reads.n else 1
    mask = np.zeros((len(probs), stride), dtype=np.uint8) if want_mask else None
    st = reads._struct()
    self._check(lib.bt2g_ungapped(self._h, C.byref(st), _ptr(probs), len(probs), _ptr(out), _ptr(mask), stride), "bt2g_ungapped")
    return out, mask


Bt2Gpu.ungapped = _ungapped


# ---- extended seed table (include/bt2g.h: bt2g_build_seed_table) -----------------------------------
EXPORTS += ["bt2g_build_seed_table"]


def _build_seed_table(self, k: int):
    """Derive the k-mer start table of the seed search from the loaded index (k = 0 drops it)."""
    self._lib.bt2g_build_seed_table.argtypes = [C.c_void_p, C.c_int]
    self._check(self._lib.bt2g_build_seed_table(self._h, int(k)), "bt2g_build_seed_table")


Bt2Gpu.build_seed_table = _build_seed_table


# ---- denser SA sample (include/bt2g.h: bt2g_build_dense_sa) ------------------------------------------
EXPORTS += ["bt2g_build_dense_sa"]


def _build_dense_sa(self, rate: int):
    """Derive offs2[row >> rate] for rows divisible by 2^rate from the loaded index (rate < 0 drops it)."""
    self._lib.bt2g_build_dense_sa.argtypes = [C.c_void_p, C.c_int]
    self._check(self._lib.bt2g_build_dense_sa(self._h, int(rate)), "bt2g_build_dense_sa")


Bt2Gpu.build_dense_sa = _build_dense_sa


# ---- SAM records (include/bt2g.h: bt2g_sam_format; host code) ----------------------------------------
EXPORTS += ["bt2g_sam_format"]


class _SamOpts(C.Structure):
    _fields_ = [("ref_names", C.POINTER(C.c_char_p)), ("n_refs", C.c_uint64), ("read_names", C.POINTER(C.c_char_p)),
                ("threads", C.c_int32), ("sc_filter_maxlen", C.c_int32), ("nceil_const", C.c_double), ("nceil_linear", C.c_double),
                ("flags", C.c_uint32), ("reserved2", C.c_uint32), ("rg_optflag", C.c_char_p)]


def sc_filter_maxlen(local: bool, sc=None) -> int:
    """longest read whose perfect score stays below the minimum score (0 in end-to-end mode); sc: a policy.Scoring (--ma / --score-min)"""
    from . import policy
    sc = sc or policy.Scoring.default(local)
    n = 0
    for ln in range(2, 200):
        if sc.perfect_score(ln) < sc.score_min().fi(ln):
            n = ln
    return n


class HostBuffers:
    """named host arrays kept from call to call.  A batch's buffers are hundreds of megabytes; memory fresh from the allocator costs a
    page fault per 4 KB and an munmap when it is dropped, so the streaming path (stream.py) reuses one set per batch in flight."""

    def __init__(self):
        self._a = {}

    def get(self, key, shape, dtype):
        shape = tuple(int(x) for x in (shape if isinstance(shape, tuple) else (shape,)))
        n = int(np.prod(shape, dtype=np.int64)) * np.dtype(dtype).itemsize
        b = self._a.get(key)
        if b is None or b.nbytes < n:
            b = self._a[key] = np.empty(n + (n >> 3) + 64, dtype=np.uint8)
        return b[:n].view(dtype).reshape(shape)


def sam_format(lib, reads: ReadBatch, res: np.ndarray, ops, ref_names, read_names=None, pairs=None, threads: int = 1,
               local: bool = False, xeq: bool = False, no_unal: bool = False, rg_id: str = None, as_bytes=False, out: HostBuffers = None,
               no_discordant: bool = False, sc=None):
    """SAM text for pipeline results (one record per read).  `lib` is the loaded libbt2g (load_library()).
    as_bytes: False -> str, True -> bytes, "view" -> a memoryview of the output buffer (no copy; with `out` given the buffer is reused
    by the next call, so the view must be consumed before it).  no_discordant: the run's --no-discordant (BT2G_SAM_NO_DISCORDANT).
    sc: the run's policy.Scoring when it is not the default one (--ma / --score-min / --n-ceil decide the YF:Z: filter tags of unaligned reads)."""
    lib.bt2g_sam_format.argtypes = [C.POINTER(_SamOpts), C.POINTER(_Reads), C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                    C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    rn = (C.c_char_p * len(ref_names))(*[x.encode() for x in ref_names])
    if isinstance(read_names, NameTable):
        ptrs = read_names.pointers()                       # no per-name Python work
        qn = C.cast(ptrs.ctypes.data, C.POINTER(C.c_char_p))
    else:
        qn = (C.c_char_p * reads.n)(*[x.encode() for x in read_names]) if read_names is not None else None
    nce = sc.n_ceil_func() if sc is not None and sc.n_ceil_over is not None else None
    opt = _SamOpts(rn, len(ref_names), qn, int(threads), sc_filter_maxlen(True, sc) if local else 0, float(nce.C) if nce else 0.0, float(nce.L) if nce else 0.0,
                   (1 if xeq else 0) | (2 if no_unal else 0) | (4 if no_discordant else 0), 0, ("RG:Z:" + rg_id).encode() if rg_id else None)
    res = np.ascontiguousarray(res, dtype=READ_RESULT)
    max_ops = 0 if ops is None else ops.shape[1]
    if ops is not None:
        ops = np.ascontiguousarray(ops, dtype=np.uint8)
    if pairs is not None:
        pairs = np.ascontiguousarray(pairs, dtype=PAIR_RESULT)
    st = reads._struct()
    need = C.c_uint64(0)
    # one formatting pass in the common case: a buffer sized from the batch (SEQ + QUAL + ~220 bytes of fields per record);
    # the call reports the size it needs (-3) when that estimate is short
    cap = int(reads.off[-1]) * 2 + reads.n * 260 + 4096 if reads.n else 4096
    alloc = (lambda c: out.get("sam", (c,), np.uint8)) if out is not None else (lambda c: np.empty(c, dtype=np.uint8))
    buf = alloc(cap)
    rc = lib.bt2g_sam_format(C.byref(opt), C.byref(st), _ptr(res), _ptr(ops), max_ops, _ptr(pairs), _ptr(buf), cap, C.byref(need))
    if rc == -3:
        cap = int(need.value)
        buf = alloc(cap)
        rc = lib.bt2g_sam_format(C.byref(opt), C.byref(st), _ptr(res), _ptr(ops), max_ops, _ptr(pairs), _ptr(buf), cap, C.byref(need))
    if rc < 0:
        raise RuntimeError(f"bt2g_sam_format failed ({rc})")
    if rc == 1:
        import warnings
        warnings.warn("bt2g_sam_format: an alignment had more edit ops than max_ops; its CIGAR / MD:Z are incomplete (align with a larger max_ops)")
    data = buf[:int(need.value)]
    if as_bytes == "view":
        return memoryview(data)
    return data.tobytes() if as_bytes else data.tobytes().decode()


EXPORTS += ["bt2g_fastq_parse", "bt2g_fastq_parse_mt"]


class NameTable:
    """read names as the parser leaves them: one NUL-terminated row of `stride` bytes per read.  Behaves like a list of str
    (decoded on access); sam_format takes it without touching the individual names."""

    def __init__(self, rows: np.ndarray):
        self.rows = np.ascontiguousarray(rows, dtype=np.uint8)

    def __len__(self):
        return self.rows.shape[0]

    def __getitem__(self, i):
        if isinstance(i, slice):
            return NameTable(self.rows[i])
        return bytes(self.rows[i]).split(b"\0", 1)[0].decode()

    def __iter__(self):
        return (self[i] for i in range(len(self)))

    def __eq__(self, other):
        return list(self) == list(other)

    def __add__(self, other):
        return NameTable(np.concatenate([self.rows, other.rows]))

    def pointers(self):
        """array of char* (one per read) into the table"""
        n, stride = self.rows.shape
        return (self.rows.ctypes.data + stride * np.arange(n, dtype=np.uint64)).astype(np.uint64)


def fastq_parse(lib, text: bytes, max_reads: int = 1 << 30, name_stride: int = 64, threads: int = 1, out: HostBuffers = None):
    """include/bt2g.h: bt2g_fastq_parse[_mt] -> (ReadBatch, names (NameTable), bytes consumed).  With `out` the arrays live in
    reused buffers: they are valid until the next call with the same `out`."""
    args = [C.c_char_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
            C.c_uint32, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.bt2g_fastq_parse.argtypes = args
    lib.bt2g_fastq_parse_mt.argtypes = args + [C.c_int]
    cap_reads = min(max_reads, text.count(b"\n") // 4 + 1)
    cap_bases = len(text)                                   # (never reached: the untouched tail costs no memory)
    alloc = out.get if out is not None else (lambda key, shape, dtype: np.empty(shape, dtype=dtype))
    seq = alloc("seq", (cap_bases,), np.uint8)
    qual = alloc("qual", (cap_bases,), np.uint8)
    off = alloc("off", (cap_reads + 1,), np.uint64)
    off[0] = 0
    names = alloc("names", (cap_reads, name_stride), np.uint8)   # (the parser defines every byte of the rows it fills)
    n, used = C.c_uint64(0), C.c_uint64(0)
    if threads > 1:
        rc = lib.bt2g_fastq_parse_mt(text, len(text), cap_reads, cap_bases, _ptr(seq), _ptr(qual), _ptr(off), _ptr(names), name_stride,
                                     C.byref(n), C.byref(used), int(threads))
    else:
        rc = lib.bt2g_fastq_parse(text, len(text), cap_reads, cap_bases, _ptr(seq), _ptr(qual), _ptr(off), _ptr(names), name_stride,
                                  C.byref(n), C.byref(used))
    if rc:
        raise RuntimeError(f"bt2g_fastq_parse failed ({rc})")
    n = int(n.value)
    nb = int(off[n])
    return ReadBatch(seq[:nb], off[:n + 1], qual[:nb]), NameTable(names[:n]), int(used.value)


EXPORTS += ["bt2g_fastq_parse_pairs_mt"]


def fastq_parse_pairs(lib, text1: bytes, text2: bytes, name_stride: int = 64, threads: int = 1, out: HostBuffers = None, max_pairs: int = None):
    """include/bt2g.h: bt2g_fastq_parse_pairs_mt -> (ReadBatch with mate 1 of pair i as read 2i and mate 2 as read 2i + 1, names
    (NameTable, same order), bytes consumed of text1, of text2).  With `out` the arrays live in reused buffers."""
    lib.bt2g_fastq_parse_pairs_mt.argtypes = [C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                                              C.POINTER(C.c_uint64), C.c_int]
    alloc = out.get if out is not None else (lambda key, shape, dtype: np.empty(shape, dtype=dtype))
    cap_bases = len(text1) + len(text2)                     # (never reached: the untouched tail costs no memory)
    # records: the last batch's count is the first guess (batches of a run look alike); an exact line count when that was short
    guess = getattr(out, "pairs_hint", None) if out is not None else None
    cap_pairs = max_pairs if max_pairs is not None else (int(guess * 1.05) + 16 if guess else min(text1.count(b"\n"), text2.count(b"\n")) // 4 + 1)
    while True:
        seq = alloc("seq", (cap_bases,), np.uint8)
        qual = alloc("qual", (cap_bases,), np.uint8)
        off = alloc("off", (2 * cap_pairs + 1,), np.uint64)
        names = alloc("names", (2 * cap_pairs, name_stride), np.uint8)
        n, u1, u2 = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        rc = lib.bt2g_fastq_parse_pairs_mt(text1, len(text1), text2, len(text2), cap_pairs, cap_bases, _ptr(seq), _ptr(qual), _ptr(off), _ptr(names),
                                           name_stride, C.byref(n), C.byref(u1), C.byref(u2), int(threads))
        if rc:
            raise RuntimeError(f"bt2g_fastq_parse_pairs_mt failed ({rc})")
        n = int(n.value)
        if max_pairs is None and guess and n == cap_pairs and (u1.value < len(text1) or u2.value < len(text2)):
            guess, cap_pairs = None, min(text1.count(b"\n"), text2.count(b"\n")) // 4 + 1     # the guess was short: parse again
            continue
        break
    if out is not None:
        out.pairs_hint = n
    nb = int(off[2 * n])
    return ReadBatch(seq[:nb], off[:2 * n + 1], qual[:nb]), NameTable(names[:2 * n]), int(u1.value), int(u2.value)

EXPORTS += ["bt2g_mapq", "bt2g_frame_mate_host", "bt2g_pe_classify_host"]


EXPORTS += ["bt2g_sam_header", "bt2g_sam_header_rg", "bt2g_align_counts_add", "bt2g_align_counts_add_ex", "bt2g_align_summary", "bt2g_index_file_open", "bt2g_index_file_desc",
            "bt2g_index_file_n_refs", "bt2g_index_file_ref_names", "bt2g_index_file_ref_lens", "bt2g_index_file_close",
            "bt2g_load_index_files_ex"]


def sam_header(lib, names, lens, pg_cl=None, rg_id=None, rg_fields=()) -> str:
    """include/bt2g.h: bt2g_sam_header / bt2g_sam_header_rg (--rg-id <id>, --rg <field> ...)."""
    if rg_id:
        lib.bt2g_sam_header_rg.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_char_p, C.c_char_p, C.c_void_p, C.c_uint64,
                                           C.POINTER(C.c_uint64)]
        rn = (C.c_char_p * len(names))(*[x.encode() for x in names])
        ln = np.ascontiguousarray(lens, dtype=np.uint64)
        rg = "\t".join(["ID:" + rg_id] + list(rg_fields)).encode()
        cl = pg_cl.encode() if pg_cl is not None else None
        need = C.c_uint64(0)
        lib.bt2g_sam_header_rg(rn, _ptr(ln), len(names), rg, cl, None, 0, C.byref(need))
        buf = C.create_string_buffer(int(need.value) + 1)
        if lib.bt2g_sam_header_rg(rn, _ptr(ln), len(names), rg, cl, buf, need.value, C.byref(need)):
            raise RuntimeError("bt2g_sam_header_rg failed")
        return buf.raw[:need.value].decode()
    lib.bt2g_sam_header.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_char_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    rn = (C.c_char_p * len(names))(*[x.encode() for x in names])
    ln = np.ascontiguousarray(lens, dtype=np.uint64)
    cl = pg_cl.encode() if pg_cl is not None else None
    need = C.c_uint64(0)
    lib.bt2g_sam_header(rn, _ptr(ln), len(names), cl, None, 0, C.byref(need))
    buf = C.create_string_buffer(int(need.value) + 1)
    rc = lib.bt2g_sam_header(rn, _ptr(ln), len(names), cl, buf, need.value, C.byref(need))
    if rc:
        raise RuntimeError(f"bt2g_sam_header failed ({rc})")
    return buf.raw[:need.value].decode()


ALIGN_COUNTS = np.dtype([(k, np.uint64) for k in ("nread", "npaired", "nunpaired", "nconcord_0", "nconcord_uni1", "nconcord_gt1",
                                                  "ndiscord", "nunp_0_0", "nunp_0_uni1", "nunp_0_gt1", "nunp_0", "nunp_uni1", "nunp_gt1")])


def align_counts_add(lib, counts, res, pairs=None, no_discordant: bool = False):
    """include/bt2g.h: bt2g_align_counts_add[_ex]; `counts` is a 1-element ALIGN_COUNTS array (None starts a new one)."""
    if counts is None:
        counts = np.zeros(1, dtype=ALIGN_COUNTS)
    lib.bt2g_align_counts_add_ex.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32]
    res = np.ascontiguousarray(res, dtype=READ_RESULT)
    if pairs is not None:
        pairs = np.ascontiguousarray(pairs, dtype=PAIR_RESULT)
    rc = lib.bt2g_align_counts_add_ex(_ptr(counts), _ptr(res), len(res), _ptr(pairs), 4 if no_discordant else 0)
    if rc:
        raise RuntimeError(f"bt2g_align_counts_add failed ({rc})")
    return counts


def align_summary(lib, counts, discord: bool = True, mixed: bool = True) -> str:
    """include/bt2g.h: bt2g_align_summary: the text bowtie2 prints on stderr at the end of a run."""
    lib.bt2g_align_summary.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    counts = np.ascontiguousarray(counts, dtype=ALIGN_COUNTS)
    need = C.c_uint64(0)
    lib.bt2g_align_summary(_ptr(counts), int(discord), int(mixed), None, 0, C.byref(need))
    buf = C.create_string_buffer(int(need.value) + 1)
    rc = lib.bt2g_align_summary(_ptr(counts), int(discord), int(mixed), buf, need.value, C.byref(need))
    if rc:
        raise RuntimeError(f"bt2g_align_summary failed ({rc})")
    return buf.raw[:need.value].decode()


class IndexFile:
    """Host image of an index on disk (include/bt2g.h: bt2g_index_file_*); no GPU involved."""

    _ARRAYS = ("plen", "rstarts", "ebwt_fw", "ebwt_bw", "ftab_fw", "eftab_fw", "ftab_bw", "eftab_bw", "offs",
               "rec_off", "rec_len", "rec_first", "ref_buf")

    def __init__(self, basename: str, offrate: int = -1):
        lib = load_library()
        self._lib = lib
        lib.bt2g_index_file_open.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_void_p), C.c_char_p, C.c_uint32]
        lib.bt2g_index_file_desc.argtypes = [C.c_void_p]
        lib.bt2g_index_file_desc.restype = C.POINTER(_IndexHost)
        lib.bt2g_index_file_n_refs.argtypes = [C.c_void_p]
        lib.bt2g_index_file_n_refs.restype = C.c_uint64
        lib.bt2g_index_file_ref_names.argtypes = [C.c_void_p]
        lib.bt2g_index_file_ref_names.restype = C.POINTER(C.c_char_p)
        lib.bt2g_index_file_ref_lens.argtypes = [C.c_void_p]
        lib.bt2g_index_file_ref_lens.restype = C.POINTER(C.c_uint64)
        lib.bt2g_index_file_close.argtypes = [C.c_void_p]
        lib.bt2g_index_file_close.restype = None
        h = C.c_void_p()
        err = C.create_string_buffer(512)
        if lib.bt2g_index_file_open(basename.encode(), int(offrate), C.byref(h), err, 512):
            raise RuntimeError(f"bt2g_index_file_open({basename}): {err.value.decode()}")
        self._h = h
        self.desc = lib.bt2g_index_file_desc(h).contents
        n = int(lib.bt2g_index_file_n_refs(h))
        names = lib.bt2g_index_file_ref_names(h)
        self.ref_names = [names[i].decode() for i in range(n)]
        lens = lib.bt2g_index_file_ref_lens(h)
        self.ref_lens = [int(lens[i]) for i in range(int(self.desc.n_pat))]

    def scalars(self) -> dict:
        d = self.desc
        out = {k: int(getattr(d, k)) for k in ("off_size", "line_rate", "off_rate", "ftab_chars", "len", "n_pat", "n_frag",
                                               "z_off_fw", "z_off_bw", "n_recs")}
        out["fchr"] = [int(x) for x in d.fchr]
        return out

    def array(self, name: str) -> np.ndarray:
        """Copy of one array of the image, typed (OFF arrays as u32/u64, byte arrays as u8)."""
        d = self.desc
        osz = int(d.off_size)
        side = 1 << int(d.line_rate)
        nsides = ((int(d.len) // 4 + 1) + (side - 4 * osz) - 1) // (side - 4 * osz)
        ftab_len = (1 << (2 * int(d.ftab_chars))) + 1
        offs_len = (int(d.len) + 1 + (1 << int(d.off_rate)) - 1) >> int(d.off_rate)
        counts = {"plen": int(d.n_pat), "rstarts": 3 * int(d.n_frag), "ftab_fw": ftab_len, "ftab_bw": ftab_len,
                  "eftab_fw": 2 * int(d.ftab_chars), "eftab_bw": 2 * int(d.ftab_chars), "offs": offs_len,
                  "rec_off": int(d.n_recs), "rec_len": int(d.n_recs)}
        p = getattr(d, name)
        p = p if isinstance(p, int) else C.cast(p, C.c_void_p).value
        if not p:
            return None
        if name in counts:
            dt = np.uint32 if osz == 4 else np.uint64
            nbytes = counts[name] * osz
        else:
            dt = np.uint8
            if name in ("ebwt_fw", "ebwt_bw"):
                nbytes = nsides * side
            elif name == "rec_first":
                nbytes = int(d.n_recs)
            else:
                rl = self.array("rec_len")
                nbytes = (int(rl.sum()) + 3) >> 2
        buf = (C.c_uint8 * nbytes).from_address(p)
        return np.frombuffer(buf, dtype=dt).copy()

    def close(self):
        if getattr(self, "_h", None):
            self._lib.bt2g_index_file_close(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- the exact search policy in waves (include/bt2g.h: bt2g_policy_align; csrc/policy_engine.cpp) ----------------------
EXPORTS += ["bt2g_policy_align", "bt2g_policy_align_k", "bt2g_policy_align_pairs_k", "bt2g_policy_backend_gpu", "bt2g_xengine_align_host"]
_CB = C.CFUNCTYPE
_vp = C.c_void_p


class _PolicyBackend(C.Structure):
    _fields_ = [("ctx", _vp),
                ("exact_sweep", _CB(C.c_int, _vp, _vp, C.c_int, C.c_int, _vp, _vp)),
                ("seed_search", _CB(C.c_int, _vp, _vp, _vp, _vp, _vp)),
                ("one_mm", _CB(C.c_int, _vp, _vp, _vp, _vp, C.c_int32, _vp, _vp)),
                ("extend_exact", _CB(C.c_int, _vp, _vp, _vp, _vp, _vp)),
                ("resolve", _CB(C.c_int, _vp, _vp, _vp, C.c_uint64, C.c_int, _vp, _vp, _vp, _vp, _vp)),
                ("get_stretch", _CB(C.c_int, _vp, _vp, _vp, _vp, C.c_uint64, C.c_int32, _vp)),
                ("ungapped", _CB(C.c_int, _vp, _vp, _vp, C.c_uint64, _vp, _vp, C.c_uint32)),
                ("dp_extend", _CB(C.c_int, _vp, _vp, _vp, C.c_uint64, C.c_int32, C.c_int32, C.c_int32, _vp, _vp, _vp, _vp)),
                ("off_size", C.c_int32), ("reserved", C.c_int32)]


class _PePolicyS(C.Structure):
    _fields_ = [("pol", C.c_int32), ("flags", C.c_int32), ("maxfrag", C.c_uint64), ("minfrag", C.c_uint64)]


class _PolicyParams(C.Structure):
    _fields_ = [("local", C.c_int32), ("paired", C.c_int32), ("seed_len", C.c_int32), ("seed_rounds", C.c_int32), ("dp_fail_streak", C.c_int32),
                ("ival_type", C.c_int32), ("ival_const", C.c_double), ("ival_coeff", C.c_double),
                ("smin_type", C.c_int32), ("smin_const", C.c_double), ("smin_coeff", C.c_double),
                ("nceil_const", C.c_double), ("nceil_coeff", C.c_double), ("khits", C.c_int64), ("mhits", C.c_int64),
                ("mmode", C.c_int32), ("all_hits", C.c_int32), ("nofw", C.c_int32), ("norc", C.c_int32), ("discord", C.c_int32),
                ("mixed", C.c_int32), ("seed", C.c_uint32), ("max_inflight", C.c_int32),
                ("match_bonus", C.c_int32), ("mmp_max", C.c_int32), ("mmp_min", C.c_int32), ("n_pen", C.c_int32),
                ("rdgap_const", C.c_int32), ("rdgap_linear", C.c_int32), ("rfgap_const", C.c_int32), ("rfgap_linear", C.c_int32),
                ("pe", _PePolicyS), ("host_threads", C.c_int32), ("reserved", C.c_int32)]


def policy_params(preset="sensitive", local=False, paired=False, seed=0, k=None, all_hits=False, mhits=50, nofw=False, norc=False,
                  discord=True, mixed=True, pe=None, sc=None, max_inflight=0, host_threads=1, seed_len=None, seed_rounds=None,
                  dp_fail_streak=None, ival=None):
    from . import policy
    if mhits < 1:
        raise ValueError("-M must be at least 1 (the reference asserts mhits > 0, bt2_search.cpp:1775)")
    pre = policy.preset(preset, local)
    if seed_len is not None:
        pre.seed_len = seed_len                    # -L
    if seed_rounds is not None:
        pre.seed_rounds = seed_rounds              # -R
    if dp_fail_streak is not None:
        pre.dp_fail_streak = dp_fail_streak        # -D
    if ival is not None:
        pre.ival = ival                            # -i
    sc = sc or policy.Scoring.default(local)
    pe = pe or policy.PairedEndPolicy(local=local)
    smin, nce = sc.score_min(), sc.n_ceil_func()
    p = _PolicyParams()
    p.local, p.paired, p.seed_len, p.seed_rounds, p.dp_fail_streak = int(local), int(paired), pre.seed_len, pre.seed_rounds, pre.dp_fail_streak
    p.ival_type, p.ival_const, p.ival_coeff = pre.ival.type, pre.ival.C, pre.ival.L
    p.smin_type, p.smin_const, p.smin_coeff = smin.type, smin.C, smin.L
    p.nceil_const, p.nceil_coeff = nce.C, nce.L
    p.khits, p.mhits = (k or 0), mhits
    p.mmode, p.all_hits = int(not (all_hits or k is not None)), int(all_hits)
    p.nofw, p.norc, p.discord, p.mixed, p.seed, p.max_inflight = int(nofw), int(norc), int(discord), int(mixed), seed, max_inflight
    p.match_bonus, p.mmp_max, p.mmp_min, p.n_pen = sc.match_bonus, sc.mmp_max, sc.mmp_min, sc.n_pen
    p.rdgap_const, p.rdgap_linear, p.rfgap_const, p.rfgap_linear = sc.rdgap_const, sc.rdgap_linear, sc.rfgap_const, sc.rfgap_linear
    p.pe.pol, p.pe.flags, p.pe.maxfrag, p.pe.minfrag = pe.pol, pe.flags(), pe.maxfrag, pe.minfrag
    p.host_threads = host_threads
    return p


def policy_align(lib, backend: "_PolicyBackend", params: "_PolicyParams", reads: ReadBatch, names, entry="bt2g_policy_align", max_ops=None):
    """include/bt2g.h: bt2g_policy_align -> (results, ops, pairs or None, (waves, backend calls, requests)).
    entry="bt2g_xengine_align_host": the fixed-memory state machine of csrc/xengine.cuh driven on the host over the same table
    (stats = units, fallbacks to the coroutine engine, requests)."""
    fn = getattr(lib, entry)
    fn.argtypes = [C.POINTER(_PolicyBackend), C.POINTER(_PolicyParams), C.POINTER(_Reads), _vp, _vp, _vp, C.c_uint32, _vp, _vp]
    n = reads.n
    max_ops = max_ops or (int(reads.lengths().max()) + 64 if n else 64)      # (more for scoring schemes with very cheap gaps)
    res = np.zeros(n, dtype=READ_RESULT)
    ops = np.zeros((max(n, 1), max_ops), dtype=np.uint8)
    pairs = np.zeros(n // 2, dtype=PAIR_RESULT) if params.paired else None
    stats = np.zeros(3, dtype=np.uint64)
    if isinstance(names, NameTable):
        keep = names.pointers()                                # (kept alive across the call)
        qn = C.cast(keep.ctypes.data, _vp)
    else:
        keep = (C.c_char_p * n)(*[x.encode() for x in names])
        qn = C.cast(keep, _vp)
    st = reads._struct()
    rc = fn(C.byref(backend), C.byref(params), C.byref(st), qn, _ptr(res), _ptr(ops), max_ops, _ptr(pairs), _ptr(stats))
    if rc:
        raise RuntimeError(f"{entry} failed ({rc})")
    return res, ops, pairs, tuple(int(x) for x in stats)


def policy_align_pairs_k(lib, backend: "_PolicyBackend", params: "_PolicyParams", reads: ReadBatch, names, max_per_pair: int):
    """include/bt2g.h: bt2g_policy_align_pairs_k (paired -k / -a) -> (results [n_pairs, max_per_pair, 2], ops [n_pairs, max_per_pair, 2,
    max_ops], pair records [n_pairs, max_per_pair], n_entries [n_pairs], truncated, stats)"""
    lib.bt2g_policy_align_pairs_k.argtypes = [C.POINTER(_PolicyBackend), C.POINTER(_PolicyParams), C.POINTER(_Reads), _vp, C.c_uint32, _vp, _vp, C.c_uint32,
                                              _vp, _vp, _vp]
    npairs = reads.n // 2
    max_ops = int(reads.lengths().max()) + 64 if reads.n else 64
    res = np.zeros((max(npairs, 1), max_per_pair, 2), dtype=READ_RESULT)
    ops = np.zeros((max(npairs, 1), max_per_pair, 2, max_ops), dtype=np.uint8)
    pairs = np.zeros((max(npairs, 1), max_per_pair), dtype=PAIR_RESULT)
    cnt = np.zeros(max(npairs, 1), dtype=np.uint32)
    stats = np.zeros(3, dtype=np.uint64)
    if isinstance(names, NameTable):
        keep = names.pointers()
        qn = C.cast(keep.ctypes.data, _vp)
    else:
        keep = (C.c_char_p * reads.n)(*[x.encode() for x in names])
        qn = C.cast(keep, _vp)
    st = reads._struct()
    rc = lib.bt2g_policy_align_pairs_k(C.byref(backend), C.byref(params), C.byref(st), qn, int(max_per_pair), _ptr(res), _ptr(ops), max_ops, _ptr(pairs),
                                       _ptr(cnt), _ptr(stats))
    if rc < 0:
        raise RuntimeError(f"bt2g_policy_align_pairs_k failed ({rc})")
    return res[:npairs], ops[:npairs], pairs[:npairs], cnt[:npairs], rc == 1, tuple(int(x) for x in stats)


def policy_align_k(lib, backend: "_PolicyBackend", params: "_PolicyParams", reads: ReadBatch, names, max_per_read: int):
    """include/bt2g.h: bt2g_policy_align_k (unpaired -k / -a) -> (results [n, max_per_read], ops [n, max_per_read, max_ops],
    n_reported [n], truncated, (waves, backend calls, requests))"""
    lib.bt2g_policy_align_k.argtypes = [C.POINTER(_PolicyBackend), C.POINTER(_PolicyParams), C.POINTER(_Reads), _vp, C.c_uint32, _vp, _vp, C.c_uint32,
                                        _vp, _vp]
    n = reads.n
    max_ops = int(reads.lengths().max()) + 64 if n else 64
    res = np.zeros((max(n, 1), max_per_read), dtype=READ_RESULT)
    ops = np.zeros((max(n, 1), max_per_read, max_ops), dtype=np.uint8)
    cnt = np.zeros(max(n, 1), dtype=np.uint32)
    stats = np.zeros(3, dtype=np.uint64)
    if isinstance(names, NameTable):
        keep = names.pointers()                                # (kept alive across the call)
        qn = C.cast(keep.ctypes.data, _vp)
    else:
        keep = (C.c_char_p * n)(*[x.encode() for x in names])
        qn = C.cast(keep, _vp)
    st = reads._struct()
    rc = lib.bt2g_policy_align_k(C.byref(backend), C.byref(params), C.byref(st), qn, max_per_read, _ptr(res), _ptr(ops), max_ops, _ptr(cnt), _ptr(stats))
    if rc < 0:
        raise RuntimeError(f"bt2g_policy_align_k failed ({rc})")
    return res[:n], ops[:n], cnt[:n], bool(rc), tuple(int(x) for x in stats)


def policy_backend_gpu(gpu: "Bt2Gpu") -> "_PolicyBackend":
    be = _PolicyBackend()
    gpu._lib.bt2g_policy_backend_gpu.argtypes = [_vp, C.POINTER(_PolicyBackend)]
    gpu._lib.bt2g_policy_backend_gpu.restype = None
    gpu._lib.bt2g_policy_backend_gpu(gpu._h, C.byref(be))
    return be


# ---- the exact search policy on the device (include/bt2g.h: bt2g_xengine_*; csrc/xengine.cuh, xengine.cu) ---------------
EXPORTS += ["bt2g_xengine_create", "bt2g_xengine_destroy", "bt2g_xengine_align", "bt2g_xengine_run_dev", "bt2g_xengine_results_dev",
            "bt2g_xengine_stage_ms", "bt2g_xengine_streams"]

XENGINE_STAGES = ("admission", "state_machine", "one_mm", "seed_search", "seed_dp", "mate_dp", "host_fallback", "total", "dp_fill", "dp_tail")
XENGINE_STATS = ("waves", "fallback_units", "seed_dps", "mate_dps", "seed_dp_cells", "mate_dp_cells", "one_mm_requests", "seed_requests")


def name_rows(names, stride=None) -> np.ndarray:
    """list of str / NameTable -> uint8 rows [n, stride], NUL-terminated"""
    if isinstance(names, NameTable):
        return names.rows
    enc = [x.encode() for x in names]
    stride = stride or (max((len(x) for x in enc), default=1) + 1)
    rows = np.zeros((len(enc), stride), dtype=np.uint8)
    for i, x in enumerate(enc):
        rows[i, :len(x)] = np.frombuffer(x, dtype=np.uint8)
    return rows


class XEngine:
    """bt2g_xengine: the reference's search policy as a device-side state machine in waves (records identical to the reference
    program's).  params: lib.policy_params(...); max_units: pairs (or reads) per call; max_len: longest read."""

    def __init__(self, gpu: "Bt2Gpu", params: "_PolicyParams", max_units: int, max_len: int):
        self.gpu, self.params, self.max_units, self.max_len = gpu, params, int(max_units), int(max_len)
        lib = gpu._lib
        lib.bt2g_xengine_create.argtypes = [_vp, C.POINTER(_PolicyParams), C.c_uint64, C.c_uint32, C.POINTER(_vp)]
        lib.bt2g_xengine_destroy.argtypes = [_vp]
        lib.bt2g_xengine_destroy.restype = None
        lib.bt2g_xengine_align.argtypes = [_vp, C.POINTER(_Reads), _vp, C.c_uint32, _vp, _vp, C.c_uint32, _vp, _vp]
        lib.bt2g_xengine_run_dev.argtypes = [_vp, _vp, _vp, _vp, C.c_uint64, _vp, C.c_uint32, _vp, _vp]
        lib.bt2g_xengine_results_dev.argtypes = [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(C.c_uint32), C.POINTER(_vp)]
        h = _vp()
        gpu._check(lib.bt2g_xengine_create(gpu._h, C.byref(params), self.max_units, self.max_len, C.byref(h)), "bt2g_xengine_create")
        self._h = h
        self.paired = bool(params.paired)
        self.max_ops = self.max_len + 80

    def align(self, reads: ReadBatch, names=None, out: "HostBuffers" = None):
        """host buffers in -> (results, ops [n, max_ops], pairs or None, stats dict); with `out` the result arrays live in reused
        buffers (valid until the next call with the same `out`)"""
        n = reads.n
        alloc = out.get if out is not None else (lambda key, shape, dtype: np.empty(shape, dtype=dtype))
        res = alloc("res", (n,), READ_RESULT)                    # (every row is overwritten by the copy back from the device)
        ops = alloc("ops", (max(n, 1), self.max_ops), np.uint8)
        pairs = alloc("pairs", (n // 2,), PAIR_RESULT) if self.paired else None
        stats = np.zeros(8, dtype=np.uint64)
        rows = None if names is None else name_rows(names)
        st = reads._struct()
        self.gpu._check(self.gpu._lib.bt2g_xengine_align(self._h, C.byref(st), _ptr(rows), 0 if rows is None else rows.shape[1], _ptr(res), _ptr(ops),
                                                         self.max_ops, _ptr(pairs), _ptr(stats)), "bt2g_xengine_align")
        return res, ops, pairs, dict(zip(XENGINE_STATS, (int(x) for x in stats)))

    def run_dev(self, d_seq: int, d_qual: int, d_off: int, n_reads: int, d_names: int = 0, name_stride: int = 0, stream: int = 0):
        """device pointers in (ints); results stay on the device (results_dev); returns the stats dict"""
        stats = np.zeros(8, dtype=np.uint64)
        self.gpu._check(self.gpu._lib.bt2g_xengine_run_dev(self._h, d_seq, d_qual, d_off, n_reads, d_names or None, name_stride, stream or None,
                                                           _ptr(stats)), "bt2g_xengine_run_dev")
        return dict(zip(XENGINE_STATS, (int(x) for x in stats)))

    def streams(self):
        """(stream, high-priority stream) of the engine as integers (cudaStream_t)"""
        a, b = _vp(), _vp()
        self.gpu._lib.bt2g_xengine_streams.argtypes = [_vp, C.POINTER(_vp), C.POINTER(_vp)]
        self.gpu._check(self.gpu._lib.bt2g_xengine_streams(self._h, C.byref(a), C.byref(b)), "bt2g_xengine_streams")
        return a.value, b.value

    def stage_ms(self):
        """device milliseconds of the last batch per stage (bt2g_xengine_stage_ms)"""
        ms = np.zeros(10, dtype=np.float32)
        n = C.c_uint64(0)
        self.gpu._lib.bt2g_xengine_stage_ms.argtypes = [_vp, _vp, C.POINTER(C.c_uint64)]
        self.gpu._check(self.gpu._lib.bt2g_xengine_stage_ms(self._h, _ptr(ms), C.byref(n)), "bt2g_xengine_stage_ms")
        self._launches = int(n.value)
        return dict(zip(XENGINE_STAGES, (float(x) for x in ms)))

    def launches(self):
        """kernels launched by the last batch (valid after stage_ms())"""
        return getattr(self, "_launches", 0)

    def results_dev(self):
        r, o, p, m = _vp(), _vp(), _vp(), C.c_uint32()
        self.gpu._lib.bt2g_xengine_results_dev(self._h, C.byref(r), C.byref(o), C.byref(m), C.byref(p))
        return r.value, o.value, int(m.value), p.value

    def close(self):
        if self._h:
            self.gpu._lib.bt2g_xengine_destroy(self._h)
            self._h = None


# ---- the whole batch loop in C++ (csrc/stream_host.cpp) --------------------------------------------------------------------
EXPORTS += ["bt2g_stream_run"]

_STREAM_ALIGN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(_Reads), C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p)
_STREAM_NEXT = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.POINTER(C.c_void_p), C.POINTER(C.c_uint64))
_STREAM_WRITE = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_uint64)
_STREAM_READ = C.CFUNCTYPE(C.c_int64, C.c_void_p, C.c_int, C.c_void_p, C.c_uint64)


class _StreamIO(C.Structure):
    _fields_ = [("user", C.c_void_p), ("next_block", _STREAM_NEXT), ("write", _STREAM_WRITE), ("read", _STREAM_READ)]


class _StreamParams(C.Structure):
    _fields_ = [("paired", C.c_int32), ("parse_threads", C.c_int32), ("format_threads", C.c_int32), ("depth", C.c_int32), ("max_units", C.c_uint64),
                ("max_len", C.c_uint32), ("max_ops", C.c_uint32), ("name_stride", C.c_uint32), ("count_flags", C.c_uint32), ("chunk_bytes", C.c_uint64),
                ("solo_engine", C.c_void_p), ("solo_max_units", C.c_uint64)]


def stream_run(lib, engines, blocks, sink, ref_names, paired: bool, max_units: int, max_len: int, max_ops: int, name_stride: int = 64,
               parse_threads: int = 2, format_threads: int = 2, depth: int = 2, local: bool = False, no_discordant: bool = False, sc=None,
               align=None, want_counts: bool = False, files=None, chunk_bytes: int = 0, solo=None, solo_max_units: int = 0):
    """include/bt2g.h: bt2g_stream_run -- FASTQ text blocks in, SAM text out, reader / engines / ordered writer overlapped in C++.
    engines: XEngine objects (their bt2g_xengine_align is the aligner), or, with `align` given, any list: align(j, ReadBatch, NameTable)
    -> (res, ops, pairs or None) is called for engine j from that engine's thread (the CPU tests' stand-ins).
    blocks: iterable of (mate-1 text, mate-2 text or None) as bytes, whole records, at most max_units reads (pairs) each -- or None with
    files = [binary file object of mate 1 (, of mate 2)] (anything with readinto: open(..., "rb"), gzip.open): the library's reader cuts the
    blocks itself, chunk_bytes of text per file at a time (the `read` callback of bt2g_stream_io).
    solo: an UNPAIRED XEngine of the same run for the pairs whose mate 2 is empty (the reference aligns their mate 1 as an unpaired read);
    with `align` given, solo=True makes the library call align(len(engines), ...) for them.
    sink(bytes) gets the records of one block (of a run of a block with solo reads), in input order.  Returns (records written, rc, counts
    or None); raises on a stage error."""
    lib.bt2g_stream_run.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int32, C.POINTER(_StreamParams), C.POINTER(_SamOpts), C.POINTER(_StreamIO),
                                    C.c_void_p, C.POINTER(C.c_uint64), C.c_char_p, C.c_uint32]
    it = iter(blocks if blocks is not None else [])
    hold, errs = [None], []

    def read(_u, mate, dst, cap):
        try:
            view = (C.c_char * cap).from_address(dst)
            return files[mate].readinto(view) or 0
        except Exception as e:
            errs.append(e)
            return -1

    def next_block(_u, t1, l1, t2, l2):
        try:
            b = next(it, None)
            if b is None:
                return 0
            hold[0] = b                                          # (the texts stay alive until the next call)
            t1[0], l1[0] = C.cast(C.c_char_p(b[0]), C.c_void_p).value, len(b[0])
            if b[1] is not None:
                t2[0], l2[0] = C.cast(C.c_char_p(b[1]), C.c_void_p).value, len(b[1])
            else:
                t2[0], l2[0] = None, 0
            return 1
        except Exception as e:                                   # (no exception may cross the C frames)
            errs.append(e)
            return -1

    def write(_u, p, n):
        try:
            sink(C.string_at(p, n))
            return 0
        except Exception as e:
            errs.append(e)
            return -1

    if align is not None:
        def cb(eng, reads, names, stride, res, ops, mo, pairs, _stats):
            try:
                r = reads.contents
                n = int(r.n_reads)
                off = np.ctypeslib.as_array(C.cast(r.off, C.POINTER(C.c_uint64)), (n + 1,)).copy()
                nb = int(off[-1])
                seq = np.ctypeslib.as_array(C.cast(r.seq, C.POINTER(C.c_uint8)), (max(nb, 1),))[:nb].copy()
                qual = np.ctypeslib.as_array(C.cast(r.qual, C.POINTER(C.c_uint8)), (max(nb, 1),))[:nb].copy()
                rows = np.ctypeslib.as_array(C.cast(names, C.POINTER(C.c_uint8)), (n * stride,)).reshape(n, stride).copy()
                rr, oo, pp = align(int(eng or 0), ReadBatch(seq, off, qual), NameTable(rows))
                rr = np.ascontiguousarray(rr, dtype=READ_RESULT)
                C.memmove(res, rr.ctypes.data, n * READ_RESULT.itemsize)
                dst = np.ctypeslib.as_array(C.cast(ops, C.POINTER(C.c_uint8)), (n * mo,)).reshape(n, mo)
                w = min(mo, oo.shape[1])
                dst[:, :w] = oo[:n, :w]
                if pp is not None and pairs:
                    pp = np.ascontiguousarray(pp, dtype=PAIR_RESULT)
                    C.memmove(pairs, pp.ctypes.data, (n // 2) * PAIR_RESULT.itemsize)
                return 0
            except Exception as e:
                errs.append(e)
                return -30
        fn = _STREAM_ALIGN(cb)
        fn_ptr = C.cast(fn, C.c_void_p)
        handles = (C.c_void_p * len(engines))(*[j if j else None for j in range(len(engines))])
    else:
        fn = None
        fn_ptr = C.cast(lib.bt2g_xengine_align, C.c_void_p)
        handles = (C.c_void_p * len(engines))(*[e._h for e in engines])
    rn = (C.c_char_p * len(ref_names))(*[x.encode() for x in ref_names])
    nce = sc.n_ceil_func() if sc is not None and sc.n_ceil_over is not None else None
    opt = _SamOpts(rn, len(ref_names), None, int(format_threads), sc_filter_maxlen(True, sc) if local else 0, float(nce.C) if nce else 0.0,
                   float(nce.L) if nce else 0.0, 4 if no_discordant else 0, 0, None)
    sp = _StreamParams(int(paired), int(parse_threads), int(format_threads), int(depth), int(max_units), int(max_len), int(max_ops), int(name_stride),
                       4 if no_discordant else 0, int(chunk_bytes), (len(engines) if align is not None else solo._h) if solo else None, int(solo_max_units))
    io = _StreamIO(None, _STREAM_NEXT(next_block), _STREAM_WRITE(write), _STREAM_READ(read) if files is not None else _STREAM_READ())
    counts = np.zeros(1, dtype=ALIGN_COUNTS) if want_counts else None
    n_reads = C.c_uint64(0)
    err = C.create_string_buffer(512)
    rc = lib.bt2g_stream_run(fn_ptr, handles, len(engines), C.byref(sp), C.byref(opt), C.byref(io), _ptr(counts), C.byref(n_reads), err, 512)
    if errs:
        raise errs[0]
    if rc < 0:
        raise RuntimeError(f"bt2g_stream_run failed ({rc}): {err.value.decode()}")
    return int(n_reads.value), rc, counts
