"""ctypes access to the oracle (TEST INFRASTRUCTURE):
  * ``Oracle``    -- oracle/_ref/libbt2oracle.so, the plain-C restatement (oracle/bt2_oracle.c)
  * ``Reference`` -- oracle/_ref/libbt2ref_{s,l}.so, the unmodified reference behind oracle/ref_glue.cpp
Both expose the same method names so tests can run one body against either.
"""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFDIR = os.path.join(ROOT, "oracle", "_ref")
OFFMASK = 0xFFFFFFFFFFFFFFFF

u64, vp, ci = C.c_uint64, C.c_void_p, C.c_int
pu64 = C.POINTER(u64)


def ref_bin(name):
    return os.path.join(REFDIR, name)


def have_reference():
    return os.path.exists(ref_bin("libbt2ref_s.so")) and os.path.exists(ref_bin("bowtie2-build-s"))


def build_oracle():
    """(Re)build the C restatement (oracle/Makefile `oracle`)."""
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "oracle"])


# ---- index files of the reference builder ----------------------------------------------------------
# The reference programs exist only where their sources were available to build oracle/_ref/.  The index
# files the tests align against do not need them: tests/golden/reference_index_digests.json holds the
# SHA-256 of every file bowtie2-build wrote for each test genome (stored by a run with the reference
# built and BT2G_RECORD_REFERENCE=1), and the project's own builder must reproduce them byte for byte.
INDEX_DIGESTS = os.path.join(ROOT, "tests", "golden", "reference_index_digests.json")
RECORD = os.environ.get("BT2G_RECORD_REFERENCE") == "1"
_INDEX_SUFFIXES = ("1", "2", "3", "4", "rev.1", "rev.2")


def _sha(data: bytes) -> str:
    return hashlib.sha256(data).hexdigest()


def _file_sha(path):
    with open(path, "rb") as f:
        return _sha(f.read())


def _index_files(base):
    ext = "bt2l" if os.path.exists(f"{base}.1.bt2l") else "bt2"
    return {s: f"{base}.{s}.{ext}" for s in _INDEX_SUFFIXES if os.path.exists(f"{base}.{s}.{ext}")}


def _load_json(path):
    if not os.path.exists(path):
        return {}
    with open(path) as f:
        return json.load(f)


def _store_json(path, key, value):
    d = _load_json(path)
    d[key] = value
    with open(path, "w") as f:
        json.dump(d, f, indent=0, sort_keys=True)
        f.write("\n")


def read_fasta(path):
    """(names, uint8 code arrays) of a FASTA file as bowtie2-build reads it: A/C/G/T (either case) -> 0..3, anything else -> N (4)"""
    names, seqs = [], []
    with open(path, "rb") as f:
        for line in f:
            line = line.rstrip(b"\r\n")
            if line.startswith(b">"):
                names.append(line[1:].decode())
                seqs.append([])
            elif seqs:
                seqs[-1].append(line)
    lut = np.full(256, 4, np.uint8)
    for i, c in enumerate(b"ACGT"):
        lut[c] = lut[c + 32] = i
    return names, [lut[np.frombuffer(b"".join(s), np.uint8)] for s in seqs]


def build_reference_index(builder, fasta, base, extra=()):
    """The index files `builder` (bowtie2-build-s / -l) writes for `fasta` at `base`.  Without the reference builder, the
    project's own builder (bowtie2_b200.index_build) writes them, and every file must hash to what the reference builder
    wrote for the same FASTA bytes and options."""
    key = " ".join([builder, *extra, _file_sha(fasta)])
    exe = ref_bin(builder)
    if os.path.exists(exe):
        subprocess.check_call([exe, "--seed", "0", "--quiet", *extra, fasta, base])
        if RECORD:
            _store_json(INDEX_DIGESTS, key, {s: _file_sha(p) for s, p in _index_files(base).items()})
        return
    want = _load_json(INDEX_DIGESTS).get(key)
    if want is None:
        raise RuntimeError(f"{exe} is not built and no digest of its output is recorded for {fasta} ({key})")
    if extra:
        raise RuntimeError(f"the project's index builder takes no bowtie2-build options ({extra})")
    import torch
    from bowtie2_b200.index_build import build_index
    names, contigs = read_fasta(fasta)
    build_index([torch.from_numpy(c) for c in contigs], names=names, off_size=8 if builder.endswith("-l") else 4,
                mirror_offs=True).write_files(base)
    got = {s: _file_sha(p) for s, p in _index_files(base).items()}
    assert got == want, f"index of {fasta}: files differ from the reference builder's ({sorted(k for k in want if got.get(k) != want[k])})"


class _Base:
    prefix = ""

    def _bind(self, lib):
        p = self.prefix
        g = lambda n: getattr(lib, p + n)
        g("open").restype = vp; g("open").argtypes = [C.c_char_p, ci, ci]
        g("close").argtypes = [vp]; g("close").restype = None
        g("scalar").restype = u64; g("scalar").argtypes = [vp, ci, ci]
        g("rank4").argtypes = [vp, ci, u64, pu64]; g("rank4").restype = None
        g("rank1").restype = u64; g("rank1").argtypes = [vp, ci, u64, ci]
        g("rowL").restype = ci; g("rowL").argtypes = [vp, ci, u64]
        g("maplf1").restype = u64; g("maplf1").argtypes = [vp, ci, u64, ci]
        g("maplf_range").argtypes = [vp, ci, u64, u64, pu64, pu64, vp]; g("maplf_range").restype = None
        g("ftab_lohi").argtypes = [vp, ci, u64, pu64, pu64]; g("ftab_lohi").restype = None
        g("get_offset").restype = u64; g("get_offset").argtypes = [vp, u64]
        g("get_stretch").argtypes = [vp, u64, C.c_int64, C.c_int64, vp]
        g("exact_sweep").restype = u64
        g("exact_sweep").argtypes = [vp, vp, ci, ci, ci, pu64, pu64]
        g("seed_search").argtypes = [vp, vp, vp, ci, ci, ci, ci, ci, ci, ci, pu64]
        self._g = g

    SCALARS = ["len", "bwt_len", "line_rate", "off_rate", "ftab_chars", "num_sides", "side_sz", "side_bwt_sz",
               "z_off", "n_pat", "n_frag", "offs_len", "ftab_len", "eftab_len", "ebwt_tot_len"]

    def scalars(self, mirror=False):
        return {k: int(self._g("scalar")(self.h, int(mirror), i)) for i, k in enumerate(self.SCALARS)}

    def rank4(self, rows, mirror=False):
        out = np.empty((len(rows), 4), dtype=np.uint64)
        buf = (u64 * 4)()
        for i, r in enumerate(rows):
            self._g("rank4")(self.h, int(mirror), int(r), buf)
            out[i] = list(buf)
        return out

    def maplf1(self, rows, chars, mirror=False):
        return np.array([self._g("maplf1")(self.h, int(mirror), int(r), int(c)) for r, c in zip(rows, chars)], dtype=np.uint64)

    def maplf_range(self, tops, nums, mirror=False):
        """Ebwt::mapLFRange for every [top, top+num): (upto[n,4], in[n,4], chars (one per row, ranges back to back))."""
        upto = np.empty((len(tops), 4), dtype=np.uint64)
        inn = np.empty((len(tops), 4), dtype=np.uint64)
        chars = np.empty(int(np.sum(np.asarray(nums, dtype=np.uint64))), dtype=np.uint8)
        u, n_, o = (u64 * 4)(), (u64 * 4)(), 0
        for i, (t, n) in enumerate(zip(tops, nums)):
            buf = np.empty(int(n), dtype=np.uint8)
            self._g("maplf_range")(self.h, int(mirror), int(t), int(n), u, n_, buf.ctypes.data_as(vp))
            upto[i], inn[i] = list(u), list(n_)
            chars[o:o + int(n)] = buf
            o += int(n)
        return upto, inn, chars

    def ftab_lohi(self, idx, mirror=False):
        out = np.empty((len(idx), 2), dtype=np.uint64)
        t, b = u64(), u64()
        for i, x in enumerate(idx):
            self._g("ftab_lohi")(self.h, int(mirror), int(x), C.byref(t), C.byref(b))
            out[i] = (t.value, b.value)
        return out

    def get_offset(self, rows):
        return np.array([self._g("get_offset")(self.h, int(r)) for r in rows], dtype=np.uint64)

    def joined_to_text(self, qlen, off, reject):
        ti, to, tl, st = u64(), u64(), u64(), ci()
        name = "joined_to_text"
        f = self._g(name)
        f.argtypes = [vp, u64, u64, ci, pu64, pu64, pu64, C.POINTER(ci)]
        ok = f(self.h, int(qlen), int(off), int(reject), C.byref(ti), C.byref(to), C.byref(tl), C.byref(st))
        return ok, ti.value, to.value, tl.value, st.value

    def get_stretch(self, tidx, off, count):
        out = np.empty(count, dtype=np.uint8)
        self._g("get_stretch")(self.h, int(tidx), int(off), int(count), out.ctypes.data_as(vp))
        return out

    def exact_sweep(self, codes, nofw=False, norc=False):
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        m, t = (u64 * 2)(), (u64 * 4)()
        nelt = self._g("exact_sweep")(self.h, codes.ctypes.data_as(vp), len(codes), int(nofw), int(norc), m, t)
        return int(nelt), list(m), list(t)

    def seed_search(self, codes, seed_len, interval, offset, max_seeds, nofw=False, norc=False, quals=None):
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        if quals is None:
            quals = np.full(len(codes), ord("I"), dtype=np.uint8)
        quals = np.ascontiguousarray(quals, dtype=np.uint8)
        out = np.zeros((2, max_seeds, 4), dtype=np.uint64)
        n = self._g("seed_search")(self.h, codes.ctypes.data_as(vp), quals.ctypes.data_as(vp), len(codes), seed_len,
                                   interval, offset, int(nofw), int(norc), max_seeds, out.ctypes.data_as(pu64))
        return n, out

    def close(self):
        if self.h:
            self._g("close")(self.h)
            self.h = None


class Oracle(_Base):
    prefix = "bt2o_"

    def __init__(self, base, mirror=True, ref=True):
        path = ref_bin("libbt2oracle.so")
        if not os.path.exists(path):
            build_oracle()
        self.lib = C.CDLL(path)
        self._bind(self.lib)
        self.h = self.lib.bt2o_open(base.encode(), int(mirror), int(ref))
        if not self.h:
            raise RuntimeError(f"oracle: cannot open index {base}")


class Reference(_Base):
    prefix = "ref_"

    def __init__(self, base, mirror=True, ref=True, large=False):
        self.lib = C.CDLL(ref_bin("libbt2ref_l.so" if large else "libbt2ref_s.so"))
        self._bind(self.lib)
        self.h = self.lib.ref_open(base.encode(), int(mirror), int(ref))
        if not self.h:
            raise RuntimeError(f"reference: cannot open index {base}")


# ---- DP through the unmodified SwAligner (oracle/ref_glue_dp.cpp) ------------------------------
def ref_dp(R, local, codes, quals, fw, tidx, tlen, rect, minsc, rndseed=1234, max_cands=1024, max_alns=32, max_edits=4096):
    """Returns dict(found, best, cands[(row,col,score)], alns[dict(score,ns,gaps,refoff,trim5,trim3,fw,edits)])."""
    i64 = C.c_int64
    L = R.lib
    L.ref_dp.argtypes = [vp, ci, vp, vp, ci, ci, u64, i64, C.POINTER(i64), i64, C.c_uint32, ci, ci, ci, vp, vp, vp, vp]
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    quals = np.ascontiguousarray(quals, dtype=np.uint8)
    r9 = (i64 * 9)(rect.refl, rect.refr, rect.refl_pretrim, rect.refr_pretrim, rect.triml, rect.trimr,
                   rect.corel, rect.corer, rect.maxgap)
    summ = np.zeros(4, np.int64)
    cands = np.zeros(3 * max_cands, np.int64)
    alns = np.zeros(8 * max_alns, np.int64)
    eds = np.zeros(4 * max_edits, np.int32)
    L.ref_dp(R.h, int(local), codes.ctypes.data_as(vp), quals.ctypes.data_as(vp), len(codes), int(fw), int(tidx),
             int(tlen), r9, int(minsc), rndseed, max_cands, max_alns, max_edits, summ.ctypes.data_as(vp),
             cands.ctypes.data_as(vp), alns.ctypes.data_as(vp), eds.ctypes.data_as(vp))
    out = {"found": int(summ[0]), "best": int(summ[1]), "ncand": int(summ[2]), "naln": int(summ[3])}
    out["cands"] = [tuple(int(x) for x in cands[3 * i:3 * i + 3]) for i in range(min(out["ncand"], max_cands))]
    al, e0 = [], 0
    for i in range(min(out["naln"], max_alns)):
        a = alns[8 * i:8 * i + 8]
        ne = int(a[6])
        al.append({"score": int(a[0]), "ns": int(a[1]), "gaps": int(a[2]), "refoff": int(a[3]), "trim5": int(a[4]),
                   "trim3": int(a[5]), "fw": int(a[7]),
                   "edits": [[int(x) for x in eds[4 * k:4 * k + 4]] for k in range(e0, e0 + ne)]})
        e0 += ne
    out["alns"] = al
    return out


class _OScoring(C.Structure):
    _fields_ = [(k, C.c_int) for k in ("match_bonus", "mmp_max", "mmp_min", "n_pen", "rdgap_const", "rdgap_linear",
                                       "rfgap_const", "rfgap_linear", "gapbar", "local")] + [("nceil_const", C.c_double), ("nceil_linear", C.c_double)]


SCORING_OVERRIDE = None      # a bowtie2_b200.policy.Scoring: non-default penalties for the oracle calls that follow


def oracle_scoring(O, local):
    O.lib.bt2o_scoring_default.argtypes = [C.POINTER(_OScoring), ci]
    sc = _OScoring()
    O.lib.bt2o_scoring_default(C.byref(sc), int(local))
    p = SCORING_OVERRIDE
    if p is not None:
        sc.match_bonus, sc.mmp_max, sc.mmp_min, sc.n_pen = p.match_bonus, p.mmp_max, p.mmp_min, p.n_pen
        sc.rdgap_const, sc.rdgap_linear, sc.rfgap_const, sc.rfgap_linear, sc.gapbar = (p.rdgap_const, p.rdgap_linear, p.rfgap_const,
                                                                                        p.rfgap_linear, p.gapbar)
        if p.n_ceil_over is not None:
            sc.nceil_const, sc.nceil_linear = float(p.n_ceil_over.C), float(p.n_ceil_over.L)
    return sc


def oracle_dp(O, local, codes, quals, fw, tidx, rect, minsc, nceil, max_cands=1024, max_alns=32, max_edits=4096, attempts=False):
    """Same outputs as ref_dp(), from the plain-C restatement (oracle/bt2_oracle.c: bt2o_dp).  attempts=True adds
    out["attempts"] = [(candidate score, alignment index or -1)], one entry per backtrace the reference would start."""
    i64 = C.c_int64
    L = O.lib
    att = None
    if attempts:
        att = np.full(3 * 4096, -1, np.int64)
        L.bt2o_dp_attempt_log.argtypes = [vp, ci]
        L.bt2o_dp_attempt_log.restype = None
        L.bt2o_dp_attempt_count.restype = ci
        L.bt2o_dp_attempt_log(att.ctypes.data_as(vp), 4096)
    L.bt2o_scoring_default.argtypes = [C.POINTER(_OScoring), ci]
    L.bt2o_dp.argtypes = [vp, C.POINTER(_OScoring), vp, vp, ci, ci, u64, i64, i64, ci, ci, ci, i64, ci, ci, ci, ci, vp, vp, vp, vp]
    sc = oracle_scoring(O, local)
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    quals = np.ascontiguousarray(quals, dtype=np.uint8)
    summ = np.zeros(4, np.int64)
    cands = np.zeros(3 * max_cands, np.int64)
    alns = np.zeros(8 * max_alns, np.int64)
    eds = np.zeros(4 * max_edits, np.int32)
    L.bt2o_dp(O.h, C.byref(sc), codes.ctypes.data_as(vp), quals.ctypes.data_as(vp), len(codes), int(fw), int(tidx),
              int(rect.refl), int(rect.refr), int(rect.triml), int(rect.corel), int(rect.corer), int(minsc), int(nceil),
              max_cands, max_alns, max_edits, summ.ctypes.data_as(vp), cands.ctypes.data_as(vp), alns.ctypes.data_as(vp),
              eds.ctypes.data_as(vp))
    out = {"found": int(summ[0]), "best": int(summ[1]), "ncand": int(summ[2]), "naln": int(summ[3])}
    out["cands"] = [tuple(int(x) for x in cands[3 * i:3 * i + 3]) for i in range(min(out["ncand"], max_cands))]
    al, e0 = [], 0
    for i in range(min(out["naln"], max_alns)):
        a = alns[8 * i:8 * i + 8]
        ne = int(a[6])
        al.append({"score": int(a[0]), "ns": int(a[1]), "gaps": int(a[2]), "refoff": int(a[3]), "trim5": int(a[4]),
                   "trim3": int(a[5]), "fw": int(a[7]),
                   "edits": [[int(x) for x in eds[4 * k:4 * k + 4]] for k in range(e0, e0 + ne)]})
        e0 += ne
    out["alns"] = al
    if attempts:
        n = int(L.bt2o_dp_attempt_count())
        assert n <= 4096
        out["attempts"] = [(int(att[3 * k]), int(att[3 * k + 1])) for k in range(n)]
        out["attempt_cands"] = [int(att[3 * k + 2]) for k in range(n)]
        L.bt2o_dp_attempt_log(None, 0)
    return out


def extend_both(X, codes, fw, off, seedlen, rng4):
    """SwDriver::extend through the reference glue (X = Reference) or the C restatement (X = Oracle)."""
    out = (u64 * 2)()
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    f = X._g("extend")
    f.argtypes = [vp, vp, ci, ci, u64, u64, u64, u64, u64, u64, pu64]
    f.restype = None
    f(X.h, codes.ctypes.data_as(vp), len(codes), int(fw), int(off), int(seedlen), int(rng4[0]), int(rng4[1]), int(rng4[2]), int(rng4[3]), out)
    return int(out[0]), int(out[1])


# ---- SeedAligner::oneMmSearch (oracle/ref_glue.cpp: ref_one_mm, oracle/bt2_oracle.c: bt2o_one_mm) ----
def _one_mm_call(fn, first, codes, quals, minsc, nofw, norc, max_hits):
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    if quals is None:
        quals = np.full(len(codes), ord("I"), dtype=np.uint8)
    quals = np.ascontiguousarray(quals, dtype=np.uint8)
    out = np.zeros((max_hits, 6), dtype=np.int64)
    fws = np.zeros(max_hits, dtype=np.int32)
    fn.restype = ci
    n = fn(*first, codes.ctypes.data_as(vp), quals.ctypes.data_as(vp), ci(len(codes)), C.c_int64(int(minsc)),
           ci(int(nofw)), ci(int(norc)), ci(max_hits), out.ctypes.data_as(vp), fws.ctypes.data_as(vp))
    assert n <= max_hits
    return [tuple(int(x) for x in out[i]) + (int(fws[i]),) for i in range(n)]


def ref_one_mm(R, local, codes, quals, minsc, nofw=False, norc=False, max_hits=256):
    """-> list of (top, bot, pos, chr, qchr, score, fw) in SeedResults::mm1EEHits() order."""
    return _one_mm_call(R.lib.ref_one_mm, (vp(R.h), ci(int(local))), codes, quals, minsc, nofw, norc, max_hits)


def oracle_one_mm(O, local, codes, quals, minsc, nofw=False, norc=False, max_hits=256):
    sc = oracle_scoring(O, local)
    return _one_mm_call(O.lib.bt2o_one_mm, (vp(O.h), C.byref(sc)), codes, quals, minsc, nofw, norc, max_hits)


# ---- SwAligner::ungappedAlign (oracle/ref_glue_dp.cpp: ref_ungapped, oracle/bt2_oracle.c: bt2o_ungapped) ----
def ref_ungapped(R, local, codes, quals, fw, tidx, off, tlen, ohang, minsc, max_edits=1024):
    """-> (rc, dict(score, refoff, trim5, trim3, ns, refns, edits=[(pos, chr, qchr, type)]))"""
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    quals = np.ascontiguousarray(quals, dtype=np.uint8)
    out8 = np.zeros(8, np.int64)
    ed = np.zeros(4 * max_edits, np.int32)
    f = R.lib.ref_ungapped
    f.restype = ci
    i64 = C.c_int64
    rc = f(vp(R.h), ci(int(local)), codes.ctypes.data_as(vp), quals.ctypes.data_as(vp), ci(len(codes)), ci(int(fw)), u64(int(tidx)),
           i64(int(off)), i64(int(tlen)), ci(int(ohang)), i64(int(minsc)), ci(max_edits), out8.ctypes.data_as(vp), ed.ctypes.data_as(vp))
    n = int(out8[6])
    return rc, dict(score=int(out8[0]), refoff=int(out8[1]), trim5=int(out8[2]), trim3=int(out8[3]), ns=int(out8[4]),
                    refns=int(out8[5]), edits=[tuple(int(x) for x in ed[4 * k:4 * k + 4]) for k in range(n)])


def oracle_ungapped(O, local, codes, quals, fw, tidx, off, tlen, ohang, minsc):
    """-> (rc, dict(score, rowi, rowf, ns, refns, nedits, mask))"""
    sc = oracle_scoring(O, local)
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    quals = np.ascontiguousarray(quals, dtype=np.uint8)
    out6 = np.zeros(6, np.int64)
    mask = np.zeros(len(codes), np.uint8)
    f = O.lib.bt2o_ungapped
    f.restype = ci
    i64 = C.c_int64
    rc = f(vp(O.h), C.byref(sc), codes.ctypes.data_as(vp), quals.ctypes.data_as(vp), ci(len(codes)), ci(int(fw)), u64(int(tidx)),
           i64(int(off)), i64(int(tlen)), ci(int(ohang)), i64(int(minsc)), out6.ctypes.data_as(vp), mask.ctypes.data_as(vp))
    return rc, dict(score=int(out6[0]), rowi=int(out6[1]), rowf=int(out6[2]), ns=int(out6[3]), refns=int(out6[4]),
                    nedits=int(out6[5]), mask=mask)


def oracle_policy_table(O, local=False, off_size=4, scoring=None):
    """bt2g_policy_backend filled with the C oracle's functions (oracle/bt2_oracle_table.c): the exact-policy engine driven on the
    CPU at C speed.  Returns (table, handle to keep alive)."""
    from bowtie2_b200.lib import _PolicyBackend
    be = _PolicyBackend()
    O.lib.bt2o_policy_table.argtypes = [vp, ci, ci, C.POINTER(_PolicyBackend)]
    O.lib.bt2o_policy_table.restype = vp
    h = O.lib.bt2o_policy_table(O.h, int(local), int(off_size), C.byref(be))
    if scoring is not None:
        O.lib.bt2o_policy_table_scoring.argtypes = [vp] + [ci] * 8
        O.lib.bt2o_policy_table_scoring.restype = None
        O.lib.bt2o_policy_table_scoring(h, scoring.match_bonus, scoring.mmp_max, scoring.mmp_min, scoring.n_pen, scoring.rdgap_const,
                                        scoring.rdgap_linear, scoring.rfgap_const, scoring.rfgap_linear)
        if scoring.n_ceil_over is not None:
            O.lib.bt2o_policy_table_nceil.argtypes = [vp, C.c_double, C.c_double]
            O.lib.bt2o_policy_table_nceil.restype = None
            O.lib.bt2o_policy_table_nceil(h, float(scoring.n_ceil_over.C), float(scoring.n_ceil_over.L))
    return be, (O, h)
