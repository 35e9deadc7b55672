#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 hot path (BASELINE.json metric: Mreads/s, 2x150 bp, 3 Gbp index).

Default workload = BASELINE.json configs[2], the configuration the metric is quoted on: synthetic 3 Gbp genome
(.bt2 index built on the GPU by bowtie2_b200.index_build, byte-identical layout to bowtie2-build-s), 2x150 bp FR
pairs (fragment ~ N(350,30)), --end-to-end --very-sensitive.  A "read" in Mreads/s is one PAIR, as in the
reference's own summary ("N reads; of these: N were paired").

The measured path is the EXACT one (`--pipeline exact`, default): the reference's search policy
(multiseedSearchWorker + SwDriver::extendSeeds[Paired]) as a device-side state machine in waves (bt2g_xengine_*,
csrc/xengine.cuh / xengine.cu) over the FM / DP kernels.  A "step" is one batch of `--batch` pairs through it:
read seeds + exactSweep at admission, then waves of {state machine step -> 1-mismatch search, (re-)seeding,
seed-extension DP, mate-finding DP} until every pair has reported.  PARITY GATE: before timing, rank 0 runs the
unmodified reference program on a FASTQ sample of the same pairs (same index files, --seed 0 --reorder) and the
engine on the same sample; the line carries "parity": {"records", "identical"} (whole SAM records: FLAG, POS,
MAPQ, CIGAR, mate fields, TLEN, AS/XS/YS/NM/MD/YT ...) and `value` is refused unless every record is identical.
`--pipeline speculative` is round 1's batch pipeline (not SAM-identical; kept as a diagnostic only).
`--workload se100` runs configs[1] (10 M x 100 bp unpaired, --sensitive) instead.

    python bench.py --gpus N --steps K --warmup W          # our arm (torchrun for N > 1)
    python bench.py --impl reference ...                    # the reference CPU bowtie2 on the host cores

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for the field definitions.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GENOME_CONTIGS, CONTIG_LEN = 24, 125_000_000
WORKLOADS = {
    # name: paired, read length, preset, default number of units (pairs / reads) resident in HBM
    "pe150": dict(paired=True, read_len=150, preset="very-sensitive", units=10_000_000,
                  label="BASELINE.json configs[2]: 2x150 bp paired, --end-to-end --very-sensitive"),
    "se100": dict(paired=False, read_len=100, preset="sensitive", units=10_000_000,
                  label="BASELINE.json configs[1]: 1x100 bp unpaired, --end-to-end --sensitive"),
    # configs[3]: --local on 300 bp reads (the i16 territory of the reference's local SSE kernel); the engine's local DP is the
    # round-1 kernel (one problem per warp, not the H-byte design) and local candidate lists overflow the unit capacities more
    # often (host fallback): measured for completeness, not tuned
    "loc300": dict(paired=False, read_len=300, preset="very-sensitive", local=True, units=1_000_000, batch=250_000,
                   label="BASELINE.json configs[3]: 1x300 bp unpaired, --local --very-sensitive-local"),
    # configs[4]'s index FORMAT and preset on one GPU: a large (.bt2l: 64-bit offsets, 128-byte sides, 64-bit RNG draws) index over
    # the 3 Gbp genome.  Not 6 Gbp: beyond 4 Gbp the bench's torch index BUILDER (tooling, not the product) is not correct yet --
    # the reference's bowtie2-align-l rejects its files -- and its suffix sort would need more than 180 GB at 6 Gbp
    "pe150l": dict(paired=True, read_len=150, preset="sensitive", units=4_000_000, large=True, genome_mbp=3000.0, seed_table=15,
                   label="BASELINE.json configs[4]'s format and preset on one GPU: .bt2l large index, 2x150 bp paired, --end-to-end --sensitive"),
}
WORKDIR = os.environ.get("BT2G_BENCH_DIR", "/dev/shm/bt2g_bench")


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------------
# synthetic data on the GPU
# ------------------------------------------------------------------------------------------------
def make_genome_gpu(torch, dev, n_contigs, contig_len, seed=20260922, repeat_fams=50, repeat_len=5000, repeat_copies=120,
                    n_gap=10_000):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    contigs = [torch.randint(0, 4, (contig_len,), dtype=torch.uint8, device=dev, generator=g) for _ in range(n_contigs)]
    rng = np.random.default_rng(seed)
    if contig_len > 4 * repeat_len:
        fams = max(1, int(repeat_fams * (n_contigs * contig_len) / 3e9))
        for _ in range(fams):
            sc, sp = int(rng.integers(0, n_contigs)), int(rng.integers(0, contig_len - repeat_len))
            seg = contigs[sc][sp:sp + repeat_len].clone()
            for _ in range(repeat_copies):
                c, p = int(rng.integers(0, n_contigs)), int(rng.integers(0, contig_len - repeat_len))
                contigs[c][p:p + repeat_len] = seg
    if contig_len > 8 * n_gap:
        for c in contigs:
            p = contig_len // 2
            c[p:p + n_gap] = 4
    return contigs


def make_reads_gpu(torch, dev, contigs, n_reads, read_len, seed=1, sub_rate=0.005, indel_frac=0.05, random_frac=0.01):
    """uint8 [n, L] codes and Phred+33 qualities on the device; reads are drawn from either strand."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    nc, clen = len(contigs), contigs[0].numel()
    genome = torch.cat(contigs)
    span = read_len + 4
    ci = torch.randint(0, nc, (n_reads,), device=dev, generator=g)
    pos = torch.randint(0, clen - span, (n_reads,), device=dev, generator=g)
    start = ci * clen + pos
    ar = torch.arange(read_len, device=dev)
    # one short indel in a fraction of reads (deletion from / insertion into the read)
    u = torch.rand(n_reads, device=dev, generator=g)
    dlen = torch.randint(1, 4, (n_reads,), device=dev, generator=g)
    ipos = torch.randint(10, read_len - 10, (n_reads,), device=dev, generator=g)
    is_del = u < indel_frac / 2
    is_ins = (u >= indel_frac / 2) & (u < indel_frac)
    shift = torch.zeros(n_reads, read_len, dtype=torch.int64, device=dev)
    after = ar[None, :] >= ipos[:, None]
    shift += (after & is_del[:, None]) * dlen[:, None]
    ins_amt = torch.clamp(ar[None, :] - ipos[:, None] + 1, min=0)
    ins_amt = torch.minimum(ins_amt, dlen[:, None])
    shift -= is_ins[:, None] * ins_amt
    idx = start[:, None] + ar[None, :] + shift
    reads = genome[idx]
    del idx, shift
    in_ins = is_ins[:, None] & after & (ar[None, :] < (ipos + dlen)[:, None])
    rnd_base = torch.randint(0, 4, (n_reads, read_len), dtype=torch.uint8, device=dev, generator=g)
    reads = torch.where(in_ins, rnd_base, reads)
    sub = (torch.rand(n_reads, read_len, device=dev, generator=g) < sub_rate) & (reads < 4)
    reads = torch.where(sub, (reads + 1 + rnd_base % 3) % 4, reads)
    randr = torch.rand(n_reads, device=dev, generator=g) < random_frac
    reads = torch.where(randr[:, None], rnd_base, reads)
    rc = torch.rand(n_reads, device=dev, generator=g) < 0.5
    comp = torch.tensor([3, 2, 1, 0, 4], dtype=torch.uint8, device=dev)
    reads = torch.where(rc[:, None], comp[reads.flip(1).long()], reads)
    q = torch.linspace(40, 20, read_len, device=dev)[None, :] + 3.0 * torch.randn(n_reads, read_len, device=dev, generator=g)
    quals = (torch.clamp(q, 2, 41).to(torch.uint8) + 33)
    del genome
    return reads.contiguous(), quals.contiguous()


def _with_errors(torch, dev, g, genome, start, read_len, sub_rate, indel_frac):
    """read_len bases starting at joined offset `start`, with substitutions and (in a fraction of reads) one short indel"""
    n = start.numel()
    ar = torch.arange(read_len, device=dev)
    u = torch.rand(n, device=dev, generator=g)
    dlen = torch.randint(1, 4, (n,), device=dev, generator=g)
    ipos = torch.randint(10, read_len - 10, (n,), device=dev, generator=g)
    is_del = u < indel_frac / 2
    is_ins = (u >= indel_frac / 2) & (u < indel_frac)
    after = ar[None, :] >= ipos[:, None]
    shift = (after & is_del[:, None]) * dlen[:, None]
    ins_amt = torch.minimum(torch.clamp(ar[None, :] - ipos[:, None] + 1, min=0), dlen[:, None])
    shift = shift - is_ins[:, None] * ins_amt
    reads = genome[start[:, None] + ar[None, :] + shift]
    del shift
    in_ins = is_ins[:, None] & after & (ar[None, :] < (ipos + dlen)[:, None])
    rnd_base = torch.randint(0, 4, (n, read_len), dtype=torch.uint8, device=dev, generator=g)
    reads = torch.where(in_ins, rnd_base, reads)
    sub = (torch.rand(n, read_len, device=dev, generator=g) < sub_rate) & (reads < 4)
    reads = torch.where(sub, (reads + 1 + rnd_base % 3) % 4, reads)
    return reads, rnd_base


def make_pairs_gpu(torch, dev, contigs, n_pairs, read_len, seed=1, sub_rate=0.005, indel_frac=0.05, random_frac=0.01,
                   ins_mean=350.0, ins_sd=30.0, chunk=1_000_000):
    """FR pairs (SURVEY.md 8d): uint8 [2n, L] codes / qualities, mate 1 at even rows, mate 2 at odd rows."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    nc, clen = len(contigs), contigs[0].numel()
    genome = torch.cat(contigs)
    comp = torch.tensor([3, 2, 1, 0, 4], dtype=torch.uint8, device=dev)
    reads = torch.empty(2 * n_pairs, read_len, dtype=torch.uint8, device=dev)
    quals = torch.empty(2 * n_pairs, read_len, dtype=torch.uint8, device=dev)
    for c0 in range(0, n_pairs, chunk):
        n = min(chunk, n_pairs - c0)
        frag = torch.clamp(ins_mean + ins_sd * torch.randn(n, device=dev, generator=g), read_len + 20, 500).long()
        ci = torch.randint(0, nc, (n,), device=dev, generator=g)
        pos = (torch.rand(n, device=dev, generator=g) * (clen - 520)).long()
        start = ci * clen + pos
        left, rnd_l = _with_errors(torch, dev, g, genome, start, read_len, sub_rate, indel_frac)
        right, rnd_r = _with_errors(torch, dev, g, genome, start + frag - read_len, read_len, sub_rate, indel_frac)
        right = comp[right.flip(1).long()]                      # mate from the fragment's right end reads inwards
        randp = torch.rand(n, device=dev, generator=g) < random_frac
        left = torch.where(randp[:, None], rnd_l, left)
        right = torch.where(randp[:, None], rnd_r, right)
        flip = torch.rand(n, device=dev, generator=g) < 0.5      # fragment taken from the reverse strand
        m1 = torch.where(flip[:, None], right, left)
        m2 = torch.where(flip[:, None], left, right)
        reads[2 * c0:2 * (c0 + n):2] = m1
        reads[2 * c0 + 1:2 * (c0 + n):2] = m2
        q = torch.linspace(40, 20, read_len, device=dev)[None, :] + 3.0 * torch.randn(2 * n, read_len, device=dev, generator=g)
        quals[2 * c0:2 * (c0 + n)] = torch.clamp(q, 2, 41).to(torch.uint8) + 33
        del left, right, rnd_l, rnd_r, m1, m2, q
    del genome
    return reads, quals


def fastq_text(reads_np, quals_np, first_id=0) -> bytes:
    """the same records as write_fastq, as bytes in memory"""
    import tempfile
    with tempfile.NamedTemporaryFile(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as f:
        write_fastq(f.name, reads_np, quals_np, first_id)
        return open(f.name, "rb").read()


def write_fastq(path, reads_np, quals_np, first_id=0):
    """fixed-width FASTQ records written as one uint8 matrix (fast)."""
    n, L = reads_np.shape
    dna = np.frombuffer(b"ACGTN", dtype=np.uint8)
    idw = 9
    rec = 2 + idw + 1 + L + 3 + L + 1
    out = np.empty((n, rec), dtype=np.uint8)
    out[:, 0] = ord("@"); out[:, 1] = ord("r")
    ids = np.arange(first_id, first_id + n)
    for k in range(idw):
        out[:, 2 + idw - 1 - k] = (ids // 10 ** k) % 10 + ord("0")
    o = 2 + idw
    out[:, o] = ord("\n"); o += 1
    out[:, o:o + L] = dna[reads_np]; o += L
    out[:, o] = ord("\n"); out[:, o + 1] = ord("+"); out[:, o + 2] = ord("\n"); o += 3
    out[:, o:o + L] = quals_np; o += L
    out[:, o] = ord("\n")
    out.tofile(path)


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the unmodified reference binary on the host cores
# ------------------------------------------------------------------------------------------------
LARGE_INDEX = False              # set by main() for a .bt2l workload: the reference's large-index binary


def ref_binary():
    if LARGE_INDEX:
        return os.path.join(ROOT, "oracle", "_ref", "bowtie2-align-l"), "bowtie2-align-l (SSE2)"
    flags = open("/proc/cpuinfo").read() if os.path.exists("/proc/cpuinfo") else ""
    v256 = os.path.join(ROOT, "oracle", "_ref", "bowtie2-align-s-v256")
    sse = os.path.join(ROOT, "oracle", "_ref", "bowtie2-align-s")
    if " avx2 " in flags and " bmi2 " in flags and " fma " in flags and os.path.exists(v256):
        return v256, "bowtie2-align-s-v256 (AVX2)"
    return sse, "bowtie2-align-s (SSE2)"


def _ref_cmd(exe, preset, threads, index_base, fq, out="/dev/null", reorder=False):
    inp = ["-1", fq[0], "-2", fq[1]] if isinstance(fq, (tuple, list)) else ["-U", fq]
    return [exe, *preset, "--seed", "0", "-p", str(threads), *(["--reorder"] if reorder else []), "-x", index_base, *inp, "-S", out]


def run_reference(index_base, fq, threads, preset, out="/dev/null", reorder=False):
    """wall seconds of one run of the unmodified reference program (index load included)"""
    exe, _ = ref_binary()
    t0 = time.time()
    subprocess.check_call(_ref_cmd(exe, preset, threads, index_base, fq, out, reorder), stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    return time.time() - t0


def reference_thread_candidates(hw_threads, cpu_quota):
    """-p values tried for the reference, on the BIG sample: the CPUs this container may actually use (cgroup quota, else
    every hardware thread), and twice / half that -- the reference does not always scale to every hardware thread."""
    base = max(1, int(round(cpu_quota))) if cpu_quota else hw_threads
    base = min(base, hw_threads)
    c = {base, min(hw_threads, 2 * base)}
    if not cpu_quota:
        c.add(max(1, base // 2))
    return sorted(c, reverse=True)


def time_reference(index_base, fq_small, fq_big, n_small, n_big, threads, preset, t_big=None):
    """reads (pairs)/s of the reference on the host cores, with index-load time removed by differencing
    two sample sizes (same command otherwise).  fq_* is a path (unpaired) or a (mate1, mate2) tuple."""
    exe, label = ref_binary()
    if not os.path.exists(exe):
        return None
    t_small = run_reference(index_base, fq_small, threads, preset)
    if t_big is None:
        t_big = run_reference(index_base, fq_big, threads, preset)
    dt = max(t_big - t_small, 1e-6)
    return {"reads_per_s": (n_big - n_small) / dt, "t_small": t_small, "t_big": t_big, "binary": label, "threads": threads}


def device_name_rows(torch, dev, first_id, n_units, mates, stride=16):
    """read-name rows as the FASTQ sample spells them ("r%09d", both mates of a pair share it), NUL-padded to `stride` bytes:
    the per-read RNG seed of the reference hashes the name (pat.cpp:45-82), so the engine gets the same names."""
    ids = torch.arange(first_id, first_id + n_units, device=dev, dtype=torch.int64)
    rows = torch.zeros(n_units, stride, dtype=torch.uint8, device=dev)
    rows[:, 0] = ord("r")
    for k in range(9):
        rows[:, 9 - k] = ((ids // 10 ** k) % 10 + ord("0")).to(torch.uint8)
    if mates == 2:
        rows = rows.repeat_interleave(2, dim=0)
    return rows.contiguous()


# ------------------------------------------------------------------------------------------------
# round 1's speculative batch pipeline (NOT SAM-identical: diagnostic only)
# ------------------------------------------------------------------------------------------------
def run_speculative(S, args):
    import torch
    import torch.distributed as dist
    from bowtie2_b200.lib import PAIR_RESULT, READ_RESULT, Pipeline, _Reads
    gpu, dev, paired, mates, B, BR, READ_LEN, nb = S.gpu, S.dev, S.paired, S.mates, S.B, S.BR, S.READ_LEN, S.nb
    wl, reads, quals, offs, rank, world, local_rank, distributed = S.wl, S.reads, S.quals, S.offs, S.rank, S.world, S.local_rank, S.distributed
    info, cores, cpu_quota, full, unit, workload, ref_preset, cpu_baseline = S.info, S.cores, S.cpu_quota, S.full, S.unit, S.workload, S.ref_preset, S.cpu_baseline
    ktab_s, sa_s, bcast_s = S.ktab_s, S.sa_s, S.bcast_s
    line = None
    # ---- our arm -----------------------------------------------------------------------------------
    pipe = Pipeline(gpu, wl["preset"], max_len=READ_LEN, max_reads=BR, row_cap=16, range_max=8, max_cands=48, max_alns=2,
                    max_probs=4 * B, both_mates=paired)
    if paired:
        pipe.enable_pairs()
    stream = torch.cuda.Stream(device=dev)       # explicit non-default stream: kernels and timing events share it
    torch.cuda.set_stream(stream)

    def step_dev(i, count=False):
        k = i % nb
        r, q = reads[k * BR:(k + 1) * BR], quals[k * BR:(k + 1) * BR]
        if paired:
            pipe.run_paired_dev(r.data_ptr(), q.data_ptr(), offs.data_ptr(), B, stream=stream.cuda_stream, count=count)
        else:
            pipe.run_dev(r.data_ptr(), q.data_ptr(), offs.data_ptr(), B, stream=stream.cuda_stream, count=count)

    def stages():
        s = pipe.stage_ms()
        if paired:
            s.update(pipe.pair_stage_ms())
        return s

    # counters (algorithmic work) from one untimed counting pass
    step_dev(0, count=True)
    torch.cuda.synchronize()
    cnt = pipe.counters()
    if paired:
        cnt.update(pipe.pair_counters())
    for i in range(args.warmup):
        step_dev(i)
    torch.cuda.synchronize()
    if distributed:
        dist.barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record(stream)
    for i in range(args.steps):
        step_dev(args.warmup + i)
    ev1.record(stream)
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    # per-stage times: re-run the steps once more, reading the stage events after each (outside the headline timing)
    names = list(stages().keys())
    stage_acc = np.zeros(len(names))
    for i in range(args.steps):
        step_dev(args.warmup + i)
        s = stages()
        stage_acc += np.array([s[k] for k in names])
    stage_ms = dict(zip(names, (stage_acc / args.steps).tolist()))
    # ---- e2e: host buffers through the C ABI (H2D of the batch + D2H of results inside the timed region)
    import ctypes as C
    nbuf = min(2, nb)
    hseq = [torch.empty(BR * READ_LEN, dtype=torch.uint8).pin_memory() for _ in range(nbuf)]
    hqual = [torch.empty(BR * READ_LEN, dtype=torch.uint8).pin_memory() for _ in range(nbuf)]
    for k in range(nbuf):
        hseq[k].copy_(reads[k * BR:(k + 1) * BR].reshape(-1)); hqual[k].copy_(quals[k * BR:(k + 1) * BR].reshape(-1))
    hoff = np.arange(0, (BR + 1) * READ_LEN, READ_LEN, dtype=np.uint64)
    hres = torch.empty(BR * READ_RESULT.itemsize, dtype=torch.uint8).pin_memory()
    hops = torch.empty(BR * pipe.max_ops, dtype=torch.uint8).pin_memory()
    hpairs = torch.empty(max(B, 1) * PAIR_RESULT.itemsize, dtype=torch.uint8).pin_memory()

    def step_host(i):
        k = i % nbuf
        st_ = _Reads(BR, hseq[k].data_ptr(), hqual[k].data_ptr(), hoff.ctypes.data)
        if paired:
            gpu._check(gpu._lib.bt2g_pipeline_run_paired_host(pipe._h, C.byref(st_), hres.data_ptr(), hops.data_ptr(), hpairs.data_ptr()),
                       "bt2g_pipeline_run_paired_host")
        else:
            gpu._check(gpu._lib.bt2g_pipeline_run_host(pipe._h, C.byref(st_), hres.data_ptr(), hops.data_ptr()), "bt2g_pipeline_run_host")

    for i in range(min(args.warmup, 3)):
        step_host(i)
    if distributed:
        dist.barrier()
    torch.cuda.synchronize()
    t_e2e0 = time.perf_counter()
    for i in range(args.steps):
        step_host(i)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t_e2e0
    res_np = np.frombuffer(hres.numpy().tobytes(), dtype=READ_RESULT)
    found = float((res_np["found"] & 0xff != 0).mean())
    overflow = int((res_np["found"] & 0x100 != 0).sum())
    conc = None
    if paired:
        pr = np.frombuffer(hpairs.numpy().tobytes(), dtype=PAIR_RESULT)
        conc = {"concordant_frac": float((pr["pair_type"] == 1).mean()), "by_mate_dp_frac": float((pr["source"] != 0).mean())}
    clk = clocks.stop() if rank == 0 else None
    # informational: host-side SAM formatting rate of the last batch's results (bt2g_sam_format on the host threads the
    # container may use); not part of `value` or `e2e` -- the records/s it sustains is the next bottleneck (DESIGN.md section 8f)
    sam_info = None
    if rank == 0:
        try:
            from bowtie2_b200.lib import ReadBatch, sam_format
            nfmt = min(BR, 200_000) // mates * mates
            kl = (args.steps - 1) % nbuf                    # the host buffers of the last timed step
            rb = ReadBatch(hseq[kl].numpy()[:nfmt * READ_LEN], hoff[:nfmt + 1], hqual[kl].numpy()[:nfmt * READ_LEN])
            res_f = np.frombuffer(hres.numpy().tobytes(), dtype=READ_RESULT)[:nfmt]
            ops_f = hops.numpy()[:nfmt * pipe.max_ops].reshape(nfmt, pipe.max_ops)
            prs_f = np.frombuffer(hpairs.numpy().tobytes(), dtype=PAIR_RESULT)[:nfmt // 2] if paired else None
            thr = int(cpu_quota) if cpu_quota else min(cores, 16)
            t_f = time.perf_counter()
            txt = sam_format(gpu._lib, rb, res_f, ops_f, [f"chr{k + 1}" for k in range(GENOME_CONTIGS)], pairs=prs_f, threads=max(thr, 1),
                             as_bytes=True)
            dt_f = time.perf_counter() - t_f
            sam_info = {"records": nfmt, "threads": max(thr, 1), "Mrecords_per_s": nfmt / dt_f / 1e6, "bytes_per_record": len(txt) / max(nfmt, 1),
                        "note": "host formatter (one pass, multi-threaded); device-side formatting is next"}
        except Exception as e:                      # never let the informational extra break the bench line
            sam_info = {"error": repr(e)[:200]}

    # max over ranks
    t = torch.tensor([ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    if distributed:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max, e2e_ms_max = float(t[0]), float(t[1])
    total_units = args.steps * B * world
    value = total_units / (ms_max / 1e3) / 1e6
    e2e_val = total_units / (e2e_ms_max / 1e3) / 1e6

    if rank == 0:
        side = info["side_sz"]
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        # dominant kernel = the stage with the largest device time
        alg_bytes = {"exact_sweep": cnt["sweep_sides"] * side, "seed_search": cnt["seed_sides"] * side,
                     "resolve": cnt["resolve_sides"] * side, "dp": cnt["dp_cells"] * 1}
        if paired:
            alg_bytes["mate_dp"] = cnt["mate_cells"] * 1
        dom = max(alg_bytes, key=lambda k: stage_ms[k])
        fm_bytes = (cnt["sweep_sides"] + cnt["seed_sides"] + cnt["resolve_sides"]) * side
        fm_ms = stage_ms["exact_sweep"] + stage_ms["seed_search"] + stage_ms["resolve"]
        dp_ms = stage_ms["dp"] + (stage_ms["mate_dp"] if paired else 0.0)
        dp_cells = cnt["dp_cells"] + (cnt["mate_cells"] if paired else 0)
        roof = {"bound": "hbm", "kernel": dom, "achieved": alg_bytes[dom] / (stage_ms[dom] / 1e3) / 1e9, "peak": peak,
                "unit": "GB/s", "traffic": None,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy)" if peaks else "fallback 6650 GB/s",
                "algorithmic_bytes_per_launch": alg_bytes[dom], "kernel_ms": stage_ms[dom],
                "fm_stages": {"achieved": fm_bytes / (fm_ms / 1e3) / 1e9, "frac": fm_bytes / (fm_ms / 1e3) / 1e9 / peak,
                              "bytes_per_read": fm_bytes / cnt["reads"]},
                "dp_gcups": dp_cells / (dp_ms / 1e3) / 1e9}
        roof["frac"] = roof["achieved"] / peak
        pipeline_desc = ("exactSweep + multiseed round 0 + resolve(all rows of ranges<=8, cap 16) + DP/backtrace per distinct diagonal"
                         + ("; then mate framing + mate-finding DP for anchors without a concordant independent mate + pair pick" if paired else ""))
        line = {"metric": "Mreads/s", "value": value, "unit": "Mreads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u64 popcount (FM rank) + s16x2 DPX (DP)", "data": "synthetic",
                "config": {"workload": workload, "full_size": full, "read_unit": unit[:-1], "mates_per_s_M": value * mates,
                           "batch": B, "preset": " ".join(ref_preset),
                           "l2": "inputs larger than L2 (random access over a %.1f GB index; a different batch each step)" % (info["device_bytes"] / 1e9),
                           "pipeline": "speculative", "pipeline_desc": pipeline_desc, "seed_table_k": args.seed_table, "seed_table_build_s": ktab_s, "dense_sa_rate": args.dense_sa, "dense_sa_build_s": sa_s, "index_bcast_s": bcast_s, "aligned_frac": found, "pairs": conc,
                           "host_threads": cores, "cgroup_cpu_quota": cpu_quota, "dp_workspace_overflows": overflow},
                "clocks": clk, "gpu_launches": pipe.kernel_launches() * args.steps,
                "e2e": {"value": e2e_val, "unit": "Mreads/s", "h2d_bytes_per_step": 2 * BR * READ_LEN + (BR + 1) * 8,
                        "d2h_bytes_per_step": BR * READ_RESULT.itemsize + BR * pipe.max_ops + (B * PAIR_RESULT.itemsize if paired else 0)},
                "roofline": roof, "stage_ms": stage_ms, "work_per_step": cnt, "sam_format_host": sam_info, "cpu_baseline": cpu_baseline}
    return line


# ------------------------------------------------------------------------------------------------
# the exact path: bt2g_xengine_* (the reference's search policy as a device-side state machine in waves)
# ------------------------------------------------------------------------------------------------
def sam_records(path):
    """(records, reference names) of a SAM file: every non-header line, and the @SQ names in order"""
    recs, names = [], []
    with open(path) as f:
        for l in f:
            if l.startswith("@"):
                if l.startswith("@SQ"):
                    names.append(l.split("\t")[1][3:])
                continue
            recs.append(l.rstrip("\n"))
    return recs, names


def parity_gate(S, eng, sam_path, n_units, B):
    """every SAM record of the reference program on the sample vs the engine's (through the host-buffer C ABI + bt2g_sam_format)"""
    from bowtie2_b200.lib import NameTable, ReadBatch, sam_format
    want, ref_names = sam_records(sam_path)
    mates, L = S.mates, S.READ_LEN
    got = []
    fallbacks = 0
    for u0 in range(0, n_units, B):
        n = min(B, n_units - u0)
        r = S.reads[u0 * mates:(u0 + n) * mates].cpu().numpy().reshape(-1)
        q = S.quals[u0 * mates:(u0 + n) * mates].cpu().numpy().reshape(-1)
        rows = S.names[u0 * mates:(u0 + n) * mates].cpu().numpy()
        batch = ReadBatch(r, np.arange(0, (n * mates + 1) * L, L, dtype=np.uint64), q)
        res, ops, pairs, st = eng.align(batch, NameTable(rows))
        fallbacks += st["fallback_units"]
        txt = sam_format(S.gpu._lib, batch, res, ops, ref_names, read_names=NameTable(rows), pairs=pairs, threads=S.fmt_threads,
                         local=bool(S.wl.get("local")))
        got.extend(txt.rstrip("\n").split("\n"))
    same = sum(1 for a, b in zip(got, want) if a == b)
    out = {"records": len(want), "identical": same if len(got) == len(want) else min(same, len(want) - 1), "units": n_units,
           "fallback_units": fallbacks,
           "against": "the unmodified reference program (oracle/_ref, --seed 0 --reorder) on the same index files and FASTQ sample; whole SAM records"}
    if out["identical"] != out["records"]:
        bad = next((i for i, (a, b) in enumerate(zip(got, want)) if a != b), None)
        if bad is not None:
            log("first differing record:\n  ours:", got[bad][:400], "\n  ref: ", want[bad][:400])
        log(f"parity: {len(got)} records of ours vs {len(want)} of the reference")
    return out


DUMP_BYTES = 60 * 10 ** 6                # array bytes of --dump-outputs: under 64 MB with the .npy headers


def dump_outputs(S, engines, parts, out_dir):
    """What the timed path handed its caller in the last timed step -- every engine's result structs, edit ops and pair records for
    its part of the batch -- as DIR/<name>.npy (float64 fields; edit ops as float32, zero past each read's nops).  Units (pairs or
    reads) past what fits DUMP_BYTES are left out by a fixed-seed sample; unit_index.npy holds the units kept."""
    import torch
    from bowtie2_b200.lib import PAIR_RESULT, READ_RESULT
    mates = S.mates
    res, ops, pairs = [], [], []
    for e, (a, b) in zip(engines, parts):
        pr, po, mo, pp = e.results_dev()
        nr = (b - a) * mates
        host = lambda ptr, nbytes: torch.as_tensor(_DevView(ptr, nbytes), device=S.dev).cpu().numpy()
        res.append(host(pr, nr * READ_RESULT.itemsize).view(READ_RESULT))
        ops.append(host(po, nr * mo).reshape(nr, mo))
        if S.paired:
            pairs.append(host(pp, (b - a) * PAIR_RESULT.itemsize).view(PAIR_RESULT))
    res, ops = np.concatenate(res), np.concatenate(ops)
    n_units = len(res) // mates
    per_unit = mates * (8 * len(READ_RESULT.names) + 4 * ops.shape[1]) + (8 * len(PAIR_RESULT.names) if S.paired else 0) + 8
    keep = min(n_units, DUMP_BYTES // per_unit)
    units = np.arange(n_units) if keep == n_units else np.sort(np.random.default_rng(0).choice(n_units, keep, replace=False))
    rows = (units[:, None] * mates + np.arange(mates)[None, :]).reshape(-1)
    res, ops = res[rows], ops[rows].astype(np.float32)
    ops[np.arange(ops.shape[1])[None, :] >= res["nops"][:, None]] = 0
    os.makedirs(out_dir, exist_ok=True)
    out = {"unit_index": units, "read_ops": ops}
    out.update({"read_" + k: res[k] for k in READ_RESULT.names if k != "pad"})
    if S.paired:
        pr = np.concatenate(pairs)[units]
        out.update({"pair_" + k: pr[k] for k in PAIR_RESULT.names})
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v if v.dtype == np.float32 else v.astype(np.float64))
    log(f"outputs of the last timed step: {keep} of {n_units} {S.unit} written to {out_dir}")


def run_exact(S, args):
    import ctypes as C
    import torch
    import torch.distributed as dist
    from bowtie2_b200.lib import PAIR_RESULT, READ_RESULT, XEngine, _Reads, policy_params
    gpu, dev, paired, mates, B, BR, L = S.gpu, S.dev, S.paired, S.mates, S.B, S.BR, S.READ_LEN
    local = bool(S.wl.get("local"))
    prm = policy_params(S.wl["preset"], local=local, paired=paired, seed=0, host_threads=S.fmt_threads)
    # E engines, each with its own stream and host thread, take the E parts of every batch: one engine's long tail of waves
    # (a few thousand repeat-rich pairs) and its per-wave host round trips overlap with the other engines' full waves
    E = max(1, min(args.engines, B))
    sub = (B + E - 1) // E                                   # units per engine and step
    parts = [(j * sub, min(B, (j + 1) * sub)) for j in range(E)]
    parts = [(a, b) for a, b in parts if b > a]
    E = len(parts)
    engines = [XEngine(gpu, prm, sub, L) for _ in range(E)]
    # the engines' own streams (normal + high priority for the small waves of a batch's tail); events are recorded on them
    streams = [torch.cuda.ExternalStream(e.streams()[0], device=dev) for e in engines]
    free_b, total_b = torch.cuda.mem_get_info(dev)
    log(f"rank {S.rank}: {E} engine(s) of {sub} {S.unit} created; HBM in use {(total_b - free_b) / 1e9:.1f} of {total_b / 1e9:.1f} GB")
    NS = S.names.shape[1]

    # ---- parity gate (rank 0, needs the reference's SAM of the sample)
    parity = None
    if S.parity_sam:
        t0 = time.time()
        parity = parity_gate(S, engines[0], S.parity_sam, S.parity_units, sub)
        log(f"parity gate: {parity['identical']} of {parity['records']} records identical ({time.time() - t0:.1f}s)")
        try:
            os.remove(S.parity_sam)
        except OSError:
            pass
    nb = S.nb
    offs_all = S.offs

    stagger = [0.0] * E                                     # seconds engine j waits before its first step of a timed run

    def run_workers(fn, n_steps, first, staggered=False):
        """fn(j, i) for engine j over steps first..first+n_steps-1, one host thread per engine; returns after all have finished.
        staggered: engine j starts stagger[j] seconds late (inside the timed region), so that the engines -- which all take the
        same time per batch and would otherwise stay in lockstep, full waves against full waves -- run one engine's sparse tail
        under another's full waves, as worker threads with their natural jitter would"""
        errs = []

        def work(j):
            try:
                torch.cuda.set_device(dev)
                if staggered and stagger[j] > 0:
                    time.sleep(stagger[j])
                for i in range(first, first + n_steps):
                    fn(j, i)
            except Exception as e:                      # surfaced below: a failed engine must fail the bench
                errs.append(e)
        th = [threading.Thread(target=work, args=(j,)) for j in range(E)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        if errs:
            raise errs[0]

    stage_acc, stat_acc, launches = {}, {}, [0]
    lock = threading.Lock()

    def step_dev(j, i, record=False):
        k = i % nb
        a, b = parts[j]
        lo, hi = (k * B + a) * mates, (k * B + b) * mates
        r, q, nm = S.reads[lo:hi], S.quals[lo:hi], S.names[lo:hi]
        st = engines[j].run_dev(r.data_ptr(), q.data_ptr(), offs_all.data_ptr(), hi - lo, nm.data_ptr(), NS, stream=0)
        if record:
            sm = engines[j].stage_ms()                 # (host-side floats the engine filled from its own CUDA events)
            with lock:
                for kk, v in st.items():
                    stat_acc[kk] = stat_acc.get(kk, 0) + v
                for kk, v in sm.items():
                    stage_acc[kk] = stage_acc.get(kk, 0.0) + v
                launches[0] += engines[j].launches()
        return st

    run_workers(step_dev, args.warmup, 0)
    torch.cuda.synchronize()
    if E > 1 and args.stagger:
        tw = time.perf_counter()
        run_workers(step_dev, 1, 0)                          # one more untimed step: the engines' batch time
        tb = time.perf_counter() - tw
        for j in range(E):
            stagger[j] = tb * j / E
    if S.distributed:
        dist.barrier()
    clocks = ClockSampler(S.local_rank)
    if S.rank == 0:
        clocks.start()
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(E)]
    torch.cuda.synchronize()
    ev0.record(streams[0])
    torch.cuda.synchronize()                          # every engine's first kernel is ordered after ev0
    run_workers(lambda j, i: step_dev(j, i, True), args.steps, args.warmup, staggered=True)
    for j in range(E):
        ev1[j].record(streams[j])
    torch.cuda.synchronize()
    ms = max(ev0.elapsed_time(e) for e in ev1)         # first start -> last engine finished, on the device clock
    if args.dump_outputs and S.rank == 0:              # (before the untimed runs below overwrite the engines' results)
        dump_outputs(S, engines, parts, args.dump_outputs)
    stage_ms = {k: v / args.steps for k, v in stage_acc.items()}
    work = {k: v / args.steps for k, v in stat_acc.items()}
    if E > 1:
        work["waves"] = work.get("waves", 0) / E       # waves per engine and step
    # one more (untimed) part of a batch through engine 0 ALONE: the DP fill kernel's launch durations without another engine's
    # kernels sharing the GPU -- the kernel's own roofline point (the timed region's sum over concurrent engines is a lower bound)
    alone = None
    if E > 1:
        st1 = step_dev(0, 0)
        sm1 = engines[0].stage_ms()
        cells1 = st1.get("seed_dp_cells", 0) + st1.get("mate_dp_cells", 0)
        if sm1.get("dp_fill", 0) > 0:
            alone = {"units": parts[0][1] - parts[0][0], "dp_cells": cells1, "fill_ms": sm1["dp_fill"], "tail_ms": sm1.get("dp_tail"),
                     "achieved": cells1 / (sm1["dp_fill"] / 1e3) / 1e9}

    # ---- e2e: host buffers through the C ABI (H2D of reads, qualities, offsets, names + D2H of result structs, edit ops, pair records)
    nbuf = min(2, nb)
    subR = sub * mates
    hseq = [[torch.empty(subR * L, dtype=torch.uint8).pin_memory() for _ in range(nbuf)] for _ in range(E)]
    hqual = [[torch.empty(subR * L, dtype=torch.uint8).pin_memory() for _ in range(nbuf)] for _ in range(E)]
    hname = [[torch.empty(subR * NS, dtype=torch.uint8).pin_memory() for _ in range(nbuf)] for _ in range(E)]
    for j, (a, b) in enumerate(parts):
        for k in range(nbuf):
            lo, hi = (k * B + a) * mates, (k * B + b) * mates
            n = (hi - lo)
            hseq[j][k][:n * L].copy_(S.reads[lo:hi].reshape(-1)); hqual[j][k][:n * L].copy_(S.quals[lo:hi].reshape(-1))
            hname[j][k][:n * NS].copy_(S.names[lo:hi].reshape(-1))
    hoff = np.arange(0, (subR + 1) * L, L, dtype=np.uint64)
    hres = [torch.empty(subR * READ_RESULT.itemsize, dtype=torch.uint8).pin_memory() for _ in range(E)]
    hops = [torch.empty(subR * engines[0].max_ops, dtype=torch.uint8).pin_memory() for _ in range(E)]
    hpairs = [torch.empty(max(sub, 1) * PAIR_RESULT.itemsize, dtype=torch.uint8).pin_memory() for _ in range(E)]
    hstats = [np.zeros(8, dtype=np.uint64) for _ in range(E)]

    def step_host(j, i):
        k = i % nbuf
        a, b = parts[j]
        st_ = _Reads((b - a) * mates, hseq[j][k].data_ptr(), hqual[j][k].data_ptr(), hoff.ctypes.data)
        gpu._check(gpu._lib.bt2g_xengine_align(engines[j]._h, C.byref(st_), hname[j][k].data_ptr(), NS, hres[j].data_ptr(), hops[j].data_ptr(),
                                               engines[j].max_ops, hpairs[j].data_ptr() if paired else None, hstats[j].ctypes.data), "bt2g_xengine_align")

    run_workers(step_host, min(args.warmup, 2), 0)
    if S.distributed:
        dist.barrier()
    torch.cuda.synchronize()
    t_e2e0 = time.perf_counter()
    run_workers(step_host, args.steps, 0, staggered=True)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t_e2e0
    res_np = np.frombuffer(hres[0].numpy().tobytes(), dtype=READ_RESULT)[:(parts[0][1] - parts[0][0]) * mates]
    found = float((res_np["found"] & 0xff != 0).mean())
    conc = None
    if paired:
        pr = np.frombuffer(hpairs[0].numpy().tobytes(), dtype=PAIR_RESULT)[:parts[0][1] - parts[0][0]]
        conc = {"concordant_frac": float((pr["pair_type"] == 1).mean())}
    clk = clocks.stop() if S.rank == 0 else None

    # ---- text to text (rank 0, informational): FASTQ bytes in host memory -> SAM bytes in host memory, the host stages (parse,
    # format) overlapped with the engines on threads (bowtie2_b200/stream.py); bounded by the host cores this container may use
    e2e_text = None
    if S.rank == 0 and not args.no_text_e2e:
        try:
            from bowtie2_b200.stream import TextAligner
            n_items = max(2, min(2 * E, nb * E))
            items = []
            for k in range(n_items):
                a, b = parts[k % E]
                lo, hi = ((k // E) * B + a) * mates, ((k // E) * B + b) * mates
                r_np, q_np = S.reads[lo:hi].cpu().numpy(), S.quals[lo:hi].cpu().numpy()
                first = (k // E) * B + a
                items.append((fastq_text(r_np[0::mates], q_np[0::mates], first), fastq_text(r_np[1::2], q_np[1::2], first) if paired else None))
            ref_names = [f"chr{k + 1}" for k in range(GENOME_CONTIGS)]
            pthr = max(1, S.fmt_threads * 3 // 8)        # (parse is the heavier host stage per thread: tools/host_text_bench.py)
            ta = TextAligner(engines, ref_names, paired, local=local, parse_threads=pthr, format_threads=max(1, S.fmt_threads - pthr - E), name_stride=NS)
            reps = max(1, (args.steps * E + n_items - 1) // n_items)
            sam_bytes = [0]

            def sink(txt):
                sam_bytes[0] += len(txt)
            ta.run((items[k % n_items] for k in range(len(ta._slots))), sink)   # warm-up: every buffer set of the stream is touched once
            sam_bytes[0] = 0
            t0 = time.perf_counter()
            recs = ta.run((items[k % n_items] for k in range(reps * n_items)), sink)
            dt = time.perf_counter() - t0
            units = recs // mates
            e2e_text = {"value": units / dt / 1e6, "unit": "Mreads/s", "units": units, "seconds": dt,
                        "fastq_bytes": sum(len(a) + (len(b) if b else 0) for a, b in items) * reps, "sam_bytes": sam_bytes[0],
                        "host_threads_parse": pthr, "host_threads_format": max(1, S.fmt_threads - pthr - E),
                        "path": "FASTQ text (host memory) -> bt2g_fastq_parse_pairs_mt / bt2g_fastq_parse_mt -> bt2g_xengine_align -> bt2g_sam_format -> SAM text (host memory, reused buffers); "
                                "stages overlapped on host threads (bowtie2_b200/stream.py)"}
        except Exception as e:                      # informational: never breaks the bench line
            e2e_text = {"error": repr(e)[:300]}

    t = torch.tensor([ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    if S.distributed:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max, e2e_ms_max = float(t[0]), float(t[1])
    total_units = args.steps * B * S.world
    value = total_units / (ms_max / 1e3) / 1e6
    e2e_val = total_units / (e2e_ms_max / 1e3) / 1e6
    if S.rank != 0:
        return None

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    # ---- roofline of the dominant hot-path kernel: the DP fill (k_dp_fill_h), timed live by the engine's own CUDA events between
    # the fill and the tail launches of every chunk.  Algorithmic bytes: ONE byte per DP cell (the H byte the fill writes for the
    # backtrace, DESIGN.md section 3) -- the kernel is bound by that write stream, not by its DPX arithmetic (profiles/README.md).
    dp_cells = work.get("seed_dp_cells", 0) + work.get("mate_dp_cells", 0)
    fill_ms, tail_ms = stage_ms.get("dp_fill", 0.0), stage_ms.get("dp_tail", 0.0)
    dpx_peak, ncu = None, {}
    try:
        for l in open(os.path.join(ROOT, "profiles", "r02_dpx_issue_rates.json")):
            r = json.loads(l)
            if r.get("op", "").startswith("VIADDMNMX.S16x2"):
                dpx_peak = r["thread_instr_per_s"]
        ncu = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_launch_summary.json")))
    except Exception:
        pass
    roof = {"bound": "hbm", "kernel": "k_dp_fill_h (seed-extension + mate-finding rectangles)", "kernel_ms": fill_ms, "peak": peak, "unit": "GB/s",
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy)" if peaks else "fallback 6650 GB/s",
            "algorithmic_bytes_per_launch": dp_cells, "achieved": dp_cells / (fill_ms / 1e3) / 1e9 if fill_ms > 0 else 0.0,
            "traffic": ncu.get("dram_bytes_per_cell", None) and ncu["dram_bytes_per_cell"] * dp_cells,
            "traffic_source": ncu.get("source"),
            "kernel_ms_note": "sum of the fill launches' CUDA-event times over the engines; with several engines their kernels time-share the GPU, so the "
                              "sum exceeds the fill's share of the wall clock and `achieved` is a lower bound; `one_engine_alone` is the same kernel on the "
                              "same data with no other engine running (one untimed part of a batch after the timed region)",
            "one_engine_alone": alone and dict(alone, frac=alone["achieved"] / peak, unit="GB/s",
                                               dpx_frac=(3.0 * alone["dp_cells"] / (alone["fill_ms"] / 1e3) / dpx_peak) if dpx_peak else None),
            "gcups_fill": dp_cells / (fill_ms / 1e3) / 1e9 if fill_ms > 0 else None,
            "gcups_fill_and_tail": dp_cells / ((fill_ms + tail_ms) / 1e3) / 1e9 if fill_ms + tail_ms > 0 else None,
            "dpx": {"thread_instr_per_cell": 3.0, "achieved_thread_instr_per_s": 3.0 * dp_cells / (fill_ms / 1e3) if fill_ms > 0 else None,
                    "peak_thread_instr_per_s": dpx_peak, "peak_source": "profiles/r02_dpx_issue_rates.json (tools/dpx_bench.cu on this pool's B200)",
                    "frac": (3.0 * dp_cells / (fill_ms / 1e3) / dpx_peak) if (dpx_peak and fill_ms > 0) else None},
            "share_of_step": {k: stage_ms.get(k, 0.0) / max(stage_ms.get("total", 1e-9), 1e-9) for k in
                              ("dp_fill", "dp_tail", "state_machine", "admission", "one_mm", "seed_search")}}
    roof["frac"] = roof["achieved"] / peak
    line = {"metric": "Mreads/s", "value": value, "unit": "Mreads/s", "n_gpus": S.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64 popcount (FM rank) + " + ("i32 (local DP)" if local else "s16x2 DPX (DP)"), "data": "synthetic",
            "config": {"workload": S.workload, "full_size": S.full, "read_unit": S.unit[:-1], "mates_per_s_M": value * mates,
                       "batch": B, "engines": E, "engine_stagger_s": stagger, "preset": " ".join(S.ref_preset),
                       "l2": "inputs larger than L2 (random access over a %.1f GB index; a different batch each step)" % (S.info["device_bytes"] / 1e9),
                       "pipeline": "exact",
                       "pipeline_desc": "the reference's search policy (multiseedSearchWorker + SwDriver::extendSeeds[Paired], per-read RNG included) as a "
                                        "device-side state machine in waves over the FM / DP kernels (bt2g_xengine_*); SAM identical to the reference program; "
                                        f"every batch is cut into {E} parts run by {E} engines on their own streams and host threads",
                       "seed_table_k": args.seed_table, "seed_table_build_s": S.ktab_s, "dense_sa_rate": args.dense_sa, "dense_sa_build_s": S.sa_s,
                       "index_bcast_s": S.bcast_s, "aligned_frac": found, "pairs": conc, "host_threads": S.cores, "cgroup_cpu_quota": S.cpu_quota},
            "parity": parity, "clocks": clk, "gpu_launches": launches[0],
            "e2e": {"value": e2e_val, "unit": "Mreads/s", "h2d_bytes_per_step": 2 * BR * L + (BR + E) * 8 + BR * NS,
                    "d2h_bytes_per_step": BR * READ_RESULT.itemsize + BR * engines[0].max_ops + (B * PAIR_RESULT.itemsize if paired else 0),
                    "path": "bt2g_xengine_align: pinned host reads / qualities / names in, result structs + edit ops + pair records out"},
            "roofline": roof, "stage_ms": stage_ms,
            "stage_ms_note": "device time per stage and step, summed over the engines (they run concurrently: the sum can exceed ms_per_step)",
            "work_per_step": work, "e2e_text": e2e_text, "cpu_baseline": S.cpu_baseline}
    if parity is not None and parity["identical"] != parity["records"]:
        line["refused"] = {"value": value, "e2e": e2e_val, "why": "parity gate: SAM records differ from the reference program's"}
        line["value"] = None
        line["e2e"]["value"] = None
    for e in engines:
        e.close()
    return line


# ------------------------------------------------------------------------------------------------
# SURVEY 8e topology: one reader deals blocks of reads to the ranks, one ordered writer collects the results (--topology dealer)
# ------------------------------------------------------------------------------------------------
class _DevView:
    """device memory owned by the engine as a torch tensor (zero copy)"""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (int(nbytes),), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


def run_dealer(S, args):
    import torch
    import torch.distributed as dist
    from bowtie2_b200.dist import deal_blocks
    from bowtie2_b200.lib import PAIR_RESULT, READ_RESULT, XEngine, policy_params
    gpu, dev, paired, mates, L = S.gpu, S.dev, S.paired, S.mates, S.READ_LEN
    blk = min(S.B, 500_000)                                   # units per dealt block
    per_rank = max(1, args.steps * (S.B // blk))
    n_blocks = per_rank * S.world
    prm = policy_params(S.wl["preset"], local=bool(S.wl.get("local")), paired=paired, seed=0, host_threads=S.fmt_threads)
    eng = XEngine(gpu, prm, blk, L)
    NS = S.names.shape[1]
    nR = blk * mates
    offs = S.offs[:nR + 1]
    block_spec = [((nR, L), torch.uint8), ((nR, L), torch.uint8), ((nR, NS), torch.uint8)]
    result_spec = [((nR * READ_RESULT.itemsize,), torch.uint8), ((nR * eng.max_ops,), torch.uint8), ((max(blk, 1) * PAIR_RESULT.itemsize,), torch.uint8)]
    resident = S.reads.shape[0] // nR                         # blocks of reads resident on the dealer, cycled

    def get_block(k):
        j = k % resident
        return S.reads[j * nR:(j + 1) * nR], S.quals[j * nR:(j + 1) * nR], S.names[j * nR:(j + 1) * nR]

    def align(t):
        r, q, nm = t
        eng.run_dev(r.data_ptr(), q.data_ptr(), offs.data_ptr(), nR, nm.data_ptr(), NS, stream=0)
        pr, po, mo, pp = eng.results_dev()
        out = [torch.as_tensor(_DevView(pr, nR * READ_RESULT.itemsize), device=dev), torch.as_tensor(_DevView(po, nR * mo), device=dev)]
        out.append(torch.as_tensor(_DevView(pp, blk * PAIR_RESULT.itemsize), device=dev) if paired else torch.zeros(result_spec[2][0], dtype=torch.uint8, device=dev))
        return tuple(out)

    # the ordered writer (rank 0): results leave for pinned host memory block by block; blocks are released in input order
    host = [torch.empty(s, dtype=d).pin_memory() for s, d in result_spec] if S.rank == 0 else None
    state = {"next": 0, "done": set(), "bytes": 0}

    def put_result(k, res):
        for h, t in zip(host, res):
            h.copy_(t, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        state["bytes"] += sum(h.numel() for h in host)
        state["done"].add(k)
        while state["next"] in state["done"]:                 # (a writer would emit block `next` here)
            state["done"].remove(state["next"]); state["next"] += 1

    # warm-up: one block per rank, then the timed deal
    sync = lambda: torch.cuda.current_stream().synchronize()      # a received block is complete before the engine's own streams read it
    deal_blocks(S.world, block_spec, result_spec, get_block, align, put_result if S.rank == 0 else None, dev, sync=sync)
    state.update(next=0, done=set(), bytes=0)
    torch.cuda.synchronize()
    if S.distributed:
        dist.barrier()
    clocks = ClockSampler(S.local_rank)
    if S.rank == 0:
        clocks.start()
    t0 = time.perf_counter()
    deal_blocks(n_blocks, block_spec, result_spec, get_block, align, put_result if S.rank == 0 else None, dev, sync=sync)
    torch.cuda.synchronize()
    if S.distributed:
        dist.barrier()
    dt = time.perf_counter() - t0
    clk = clocks.stop() if S.rank == 0 else None
    eng.close()
    if S.rank != 0:
        return None
    assert state["next"] == n_blocks
    value = n_blocks * blk / dt / 1e6
    return {"metric": "Mreads/s", "value": value, "unit": "Mreads/s", "n_gpus": S.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64 popcount (FM rank) + s16x2 DPX (DP)", "data": "synthetic",
            "config": {"workload": S.workload, "full_size": S.full, "read_unit": S.unit[:-1], "block": blk, "blocks": n_blocks,
                       "topology": "dealer: rank 0 holds the reads and deals blocks round-robin over NCCL send / recv, every rank aligns its blocks with one "
                                   "engine, the results return to rank 0 and leave in block order for pinned host memory (SURVEY 8e: one reader, one ordered writer)",
                       "pipeline": "exact", "preset": " ".join(S.ref_preset)},
            "clocks": clk, "gpu_launches": None,
            "e2e": {"value": value, "unit": "Mreads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": state["bytes"] // max(args.steps, 1),
                    "path": "device-resident reads on the dealer -> NCCL -> engines -> NCCL -> pinned host results on the dealer"},
            "roofline": None, "cpu_baseline": S.cpu_baseline}


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pipeline", default="exact", choices=["exact", "speculative"])
    ap.add_argument("--workload", default="pe150", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=1_000_000, help="reads (pairs for a paired workload) per step")
    ap.add_argument("--topology", default="shard", choices=["shard", "dealer"],
                    help="shard (default): every rank aligns its own resident reads; dealer: rank 0 deals blocks to the ranks and collects the results in order")
    ap.add_argument("--no-stagger", dest="stagger", action="store_false",
                    help="start the engines of a timed run together instead of 1/E of a batch time apart")
    ap.add_argument("--engines", type=int, default=2, help="exact pipeline: engines (streams + host threads) that share every batch")
    ap.add_argument("--genome-mbp", type=float, default=0.0,
                    help="debug only: another genome size (0 = the workload's: 3000; any other value is NOT the BASELINE config)")
    ap.add_argument("--reads", type=int, default=0, help="reads (pairs) resident in HBM (0 = the workload's default)")
    ap.add_argument("--seed-table", type=int, default=-1,
                    help="k of the extended seed table derived from the index at load time (0 = off; results are identical)")
    ap.add_argument("--dense-sa", type=int, default=0,
                    help="rate of the denser SA sample derived from the index at load time (0 = full suffix array, -1 = off)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the reference runs (no cpu_baseline, no parity gate)")
    ap.add_argument("--no-text-e2e", action="store_true", help="skip the informational FASTQ-text -> SAM-text measurement")
    ap.add_argument("--cpu-sample", type=int, default=0, help="reads (pairs) in the CPU baseline / parity sample (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step to DIR/<name>.npy (exact pipeline, shard topology)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.pipeline != "exact" or args.topology != "shard" or args.impl != "ours"):
        ap.error("--dump-outputs needs --impl ours --pipeline exact --topology shard")
    wl = WORKLOADS[args.workload]
    paired, READ_LEN = wl["paired"], wl["read_len"]
    if args.reads <= 0:
        args.reads = wl["units"]
    wl_mbp = wl.get("genome_mbp", GENOME_CONTIGS * CONTIG_LEN / 1e6)
    if args.genome_mbp <= 0:
        args.genome_mbp = wl_mbp
    if args.seed_table < 0:
        args.seed_table = wl.get("seed_table", 16)
    global LARGE_INDEX
    LARGE_INDEX = bool(wl.get("large"))
    mates = 2 if paired else 1
    ref_preset = ("--local", "--" + wl["preset"] + "-local") if wl.get("local") else ("--end-to-end", "--" + wl["preset"])
    if wl.get("batch") and args.batch == 1_000_000:
        args.batch = wl["batch"]

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference" and rank != 0:
        return 0
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    distributed = world > 1 and args.impl == "ours"
    if distributed:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"       # keep stdout to the single JSON line
        dist.init_process_group("nccl", device_id=dev)

    from bowtie2_b200 import Bt2Gpu
    from bowtie2_b200.index_build import build_index

    class S:                                   # what the arms share
        pass
    S.wl, S.paired, S.READ_LEN, S.mates, S.ref_preset = wl, paired, READ_LEN, mates, ref_preset
    S.rank, S.world, S.local_rank, S.dev, S.distributed = rank, world, local_rank, dev, distributed
    full = abs(args.genome_mbp - wl_mbp) < 1e-6 and args.reads >= wl["units"]
    contig_len = int(args.genome_mbp * 1e6 / GENOME_CONTIGS)
    unit = "pairs" if paired else "reads"
    workload = (f"{wl['label']}: synthetic {GENOME_CONTIGS * contig_len / 1e9:.2f} Gbp genome {'.bt2l' if LARGE_INDEX else '.bt2'} index, "
                f"{args.reads / 1e6:g}M {'2x' if paired else '1x'}{READ_LEN} bp {unit} resident in HBM")
    hw_threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:                                   # container CPU quota, if any (explains where the reference stops scaling)
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        cpu_quota = None if q == "max" else float(q) / float(per)
    except Exception:
        cpu_quota = None
    S.full, S.unit, S.workload, S.cores, S.cpu_quota = full, unit, workload, hw_threads, cpu_quota
    S.fmt_threads = max(1, min(hw_threads, int(cpu_quota) if cpu_quota else 16))

    # ---- setup (untimed): genome, index (built once on rank 0, NCCL-broadcast to the others), reads
    t0 = time.time()
    contigs = make_genome_gpu(torch, dev, GENOME_CONTIGS, contig_len)
    need_files = args.impl == "reference" or (rank == 0 and not args.no_cpu_baseline)
    built = None
    if rank == 0 or not distributed:
        built = build_index(contigs, off_size=8 if LARGE_INDEX else 4)
        torch.cuda.synchronize()
        log(f"rank {rank}: index built in {time.time() - t0:.1f}s (len={built.len})")
    index_base = os.path.join(WORKDIR, "idx")
    if need_files:
        os.makedirs(WORKDIR, exist_ok=True)
        built.write_files(index_base)
        log(f"index files written to {index_base}.*.{'bt2l' if LARGE_INDEX else 'bt2'}")
    if paired:
        reads, quals = make_pairs_gpu(torch, dev, contigs, args.reads, READ_LEN, seed=1 + rank)
    else:
        reads, quals = make_reads_gpu(torch, dev, contigs, args.reads, READ_LEN, seed=1 + rank)
    del contigs
    S.reads, S.quals = reads, quals
    S.B = B = min(args.batch, args.reads)          # units (pairs / reads) per step
    S.nb = args.reads // B
    S.BR = BR = B * mates                            # reads per step
    S.offs = torch.arange(0, (BR + 1) * READ_LEN, READ_LEN, dtype=torch.int64, device=dev)

    # ---- CPU baseline / reference arm: the unmodified reference program on the same index files and a FASTQ sample ------------
    S.cpu_baseline, S.parity_sam, S.parity_units = None, None, 0
    if need_files and os.path.exists(ref_binary()[0]):
        n_big = args.cpu_sample or int(min(args.reads, 400_000 if paired else 1_000_000))
        n_small = max(n_big // 10, 1000)
        r_np = reads[:n_big * mates].cpu().numpy(); q_np = quals[:n_big * mates].cpu().numpy()
        if paired:
            fq_big = (os.path.join(WORKDIR, "big_1.fq"), os.path.join(WORKDIR, "big_2.fq"))
            fq_small = (os.path.join(WORKDIR, "small_1.fq"), os.path.join(WORKDIR, "small_2.fq"))
            for m in range(2):
                write_fastq(fq_big[m], r_np[m::2], q_np[m::2])
                write_fastq(fq_small[m], r_np[m:2 * n_small:2], q_np[m:2 * n_small:2])
        else:
            fq_big, fq_small = os.path.join(WORKDIR, "big.fq"), os.path.join(WORKDIR, "small.fq")
            write_fastq(fq_big, r_np, q_np)
            write_fastq(fq_small, r_np[:n_small], q_np[:n_small])
        del r_np, q_np
        # -p: chosen on the BIG sample among the CPUs this container may use (quota) and twice that
        t_big, threads = None, hw_threads
        for p in reference_thread_candidates(hw_threads, cpu_quota):
            dt = run_reference(index_base, fq_big, p, ref_preset)
            log(f"reference -p {p}: {dt:.2f}s for {n_big} {unit}")
            if t_big is None or dt < t_big:
                t_big, threads = dt, p
        sample = (f"{{}} {unit}: difference of a {n_big}- and a {n_small}-{unit[:-1]} run of {{}} {' '.join(ref_preset)} -p {threads} "
                  f"(fastest of -p {reference_thread_candidates(hw_threads, cpu_quota)} on the {n_big}-{unit[:-1]} sample; {hw_threads} hardware threads, "
                  f"cgroup quota {cpu_quota}; index load cancels{{}})")
        if args.impl == "reference":
            per, t_start = [], time.time()
            for s in range(args.warmup + args.steps):
                r = time_reference(index_base, fq_small, fq_big, n_small, n_big, threads, ref_preset)
                if s >= args.warmup or not per:
                    per.append(r)
                if time.time() - t_start > 150:      # keep the whole run within a few minutes
                    break
            rps = float(np.median([p["reads_per_s"] for p in per]))
            val = rps / 1e6
            line = {"metric": "Mreads/s", "value": val, "unit": "Mreads/s", "n_gpus": 0, "steps": len(per), "warmup": args.warmup,
                    "ms_per_step": 1e3 * (n_big - n_small) / rps, "higher_is_better": True, "scaling": "weak",
                    "vs_baseline": None, "dtype": "u8/i16 (SSE/AVX2 striped DP), u64 popcount FM", "data": "synthetic",
                    "impl": "reference",
                    "config": {"workload": workload, "full_size": full, "read_unit": unit[:-1], "preset": " ".join(ref_preset),
                               "host_threads": hw_threads, "cgroup_cpu_quota": cpu_quota},
                    "cpu_baseline": {"value": val, "unit": "Mreads/s", "cores": threads, "kind": "reference",
                                     "sample": sample.format(n_big - n_small, per[0]["binary"], "")},
                    "e2e": {"value": val, "unit": "Mreads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
            print(json.dumps(line))
            shutil.rmtree(WORKDIR, ignore_errors=True)
            return 0
        r = time_reference(index_base, fq_small, fq_big, n_small, n_big, threads, ref_preset, t_big=t_big)
        S.cpu_baseline = {"value": r["reads_per_s"] / 1e6, "unit": "Mreads/s", "cores": threads, "kind": "reference",
                          "sample": sample.format(n_big - n_small, r["binary"], f"; {r['t_big']:.1f}s and {r['t_small']:.1f}s wall")}
        log("cpu baseline:", S.cpu_baseline)
        if args.pipeline == "exact":
            S.parity_sam, S.parity_units = WORKDIR.rstrip("/") + ".parity.sam", n_big
            run_reference(index_base, fq_big, threads, ref_preset, out=S.parity_sam, reorder=True)
            shutil.rmtree(WORKDIR, ignore_errors=True)
        else:
            shutil.rmtree(WORKDIR, ignore_errors=True)
    elif args.impl == "reference":
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/bowtie2-align-s not built"}))
        return 0

    # ---- our arm: the index in HBM (+ the acceleration structures derived from it) ---------------------------------------------
    S.gpu = gpu = Bt2Gpu(local_rank)
    S.bcast_s = 0.0
    if distributed:
        # single broadcast of every index array from rank 0 (SURVEY.md section 8e) over NCCL / NVLink
        from bowtie2_b200.dist import broadcast_index
        torch.cuda.synchronize(); dist.barrier()
        tb = time.time()
        desc, tensors = broadcast_index(built, 0, dev)
        torch.cuda.synchronize(); dist.barrier()
        S.bcast_s = time.time() - tb
        gpu.load_index_device(desc, keep=tensors)
    else:
        gpu.load_index_device(built.device_desc(dev), keep=built)
    S.info = info = gpu.info()
    S.ktab_s = 0.0
    if args.seed_table > info["ftab_chars"]:
        torch.cuda.synchronize(); tk = time.time()
        gpu.build_seed_table(args.seed_table)
        S.ktab_s = time.time() - tk
        log(f"rank {rank}: {args.seed_table}-mer seed table built in {S.ktab_s:.2f}s")
    S.sa_s = 0.0
    if 0 <= args.dense_sa < info["off_rate"]:
        torch.cuda.synchronize(); tk = time.time()
        gpu.build_dense_sa(args.dense_sa)
        S.sa_s = time.time() - tk
        log(f"rank {rank}: SA sample of rate {args.dense_sa} built in {S.sa_s:.2f}s")
    S.names = device_name_rows(torch, dev, 0, args.reads, mates)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()                 # the genome / index-builder temporaries torch still caches: the engines allocate with cudaMalloc
    log(f"rank {rank}: setup {time.time() - t0:.1f}s, index {info['device_bytes'] / 1e9:.2f} GB in HBM")

    if args.topology == "dealer":
        line = run_dealer(S, args)
    else:
        line = run_exact(S, args) if args.pipeline == "exact" else run_speculative(S, args)
    if rank == 0:
        print(json.dumps(line))
    shutil.rmtree(WORKDIR, ignore_errors=True) if rank == 0 else None
    if distributed:
        dist.barrier()
        dist.destroy_process_group()
    return 0 if (line is None or line.get("value") is not None) else 1


if __name__ == "__main__":
    sys.exit(main())
