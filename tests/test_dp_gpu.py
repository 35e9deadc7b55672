"""GPU parity for K3: the CUDA DP (fill + gather + backtrace) through the C ABI vs the unmodified
reference SwAligner (oracle/_ref glue): found/best, the full candidate list, every alignment's
score / offset / gaps / Ns and its edit list."""
import re

import numpy as np
import pytest

from bowtie2_b200 import policy, synth
from bowtie2_b200.lib import DP_PROBLEM, ReadBatch, ops_to_edits
from oracle_lib import Reference, have_reference, ref_dp

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]


def _problems(genome, reads, truth, sc, jitter_rng, minsc_bump=0):
    """One seed-extension DP per alignable read, framed as SwDriver::extendSeeds would
    (aligner_sw_driver.cpp:1185-1283), with the seed diagonal jittered by a few bases."""
    probs, meta = [], []
    for i, (r, (c, p, strand)) in enumerate(zip(reads, truth)):
        if c < 0:
            c, p, strand = 0, int(jitter_rng.integers(0, len(genome[0]) - len(r))), 1
        rdlen = len(r)
        minsc = sc.min_score(rdlen) + minsc_bump
        if minsc > sc.perfect_score(rdlen):
            continue
        off = p + int(jitter_rng.integers(-3, 4))
        tlen = len(genome[c])
        found, rect = policy.frame_seed_extension_rect(off, rdlen, tlen, sc.max_read_gaps(minsc, rdlen),
                                                       sc.max_ref_gaps(minsc, rdlen), sc.n_ceil(rdlen))
        if not found:
            continue
        probs.append((i, 1 if strand > 0 else 0, c, rect.refl, rect.refr, rect.triml, rect.corel, rect.corer,
                      minsc, sc.n_ceil_raw(rdlen), 0))
        meta.append((tlen, rect, minsc))
    return np.array(probs, dtype=DP_PROBLEM), meta


def _check(gpu, R, genome, reads, quals, probs, meta, local=False):
    batch = ReadBatch.from_list(reads, quals)
    summ, cands, alns, ops = gpu.dp_extend(batch, probs, max_cands=8192 if local else 256, max_alns=24 if local else 8,
                                           max_ops=int(batch.lengths().max()) + 80)
    nfound = naln = ngap = 0
    for k, pr in enumerate(probs):
        tlen, rect, minsc = meta[k]
        i = int(pr["read_idx"])
        want = ref_dp(R, local, reads[i], quals[i], int(pr["fw"]), int(pr["tidx"]), tlen, rect, minsc, max_cands=16384, max_alns=64, max_edits=16384)
        s = summ[k]
        assert s["flags"] == 0, (k, s)
        assert bool(s["found"]) == bool(want["found"]), (k, s, want["found"], want["best"])
        if not want["found"]:
            # below minsc the reference's number is a saturated 8/16-bit value (0xff-biased u8 clamps
            # at -255, aligner_swsse_ee_u8.cpp:1119-1131); only "not found" is comparable
            assert s["best"] < minsc
            continue
        nfound += 1
        assert s["best"] == want["best"]
        assert s["ncand"] == want["ncand"]
        got_c = [(int(c["row"]), int(c["col"]), int(c["score"])) for c in cands[k][:s["ncand"]]]
        assert got_c == want["cands"], (k, got_c[:5], want["cands"][:5])
        assert s["naln"] == want["naln"], (k, s["naln"], want["naln"])
        for a_i, wa in enumerate(want["alns"]):
            a = alns[k][a_i]
            assert (int(a["score"]), int(a["ns"]), int(a["gaps"])) == (wa["score"], wa["ns"], wa["gaps"]), (k, a, wa)
            assert int(pr["refl"]) + int(a["col0"]) == wa["refoff"], (k, a, wa)
            ed = ops_to_edits(ops[k][a_i], int(a["nops"]), reads[i], bool(pr["fw"]), int(a["row0"]), int(a["trim_end"]))
            t5, t3 = (int(a["trim_beg"]), int(a["trim_end"])) if pr["fw"] else (int(a["trim_end"]), int(a["trim_beg"]))
            assert (t5, t3) == (wa["trim5"], wa["trim3"]), (k, a, wa)
            assert ed == wa["edits"], (k, a_i, ed, wa["edits"])
            naln += 1
            ngap += wa["gaps"] > 0
    return nfound, naln, ngap


@pytest.mark.skipif(not have_reference(), reason="oracle/_ref not built")
@pytest.mark.parametrize("rdlen,sub,indel", [(100, 0.01, 0.002), (150, 0.02, 0.004), (50, 0.01, 0.0), (250, 0.01, 0.003), (33, 0.03, 0.01),
                                             (128, 0.01, 0.003), (129, 0.02, 0.003), (180, 0.01, 0.004), (200, 0.015, 0.003)])
def test_dp_e2e_matches_reference(gpu, synth_index, synth_genome, rdlen, sub, indel):
    gpu.load_index_files(synth_index)
    gpu.set_scoring(local=False)
    R = Reference(synth_index)
    sc = policy.Scoring.default(False)
    reads, quals, truth = synth.make_reads(synth_genome, 250, rdlen, seed=rdlen, sub_rate=sub, indel_rate=indel, random_frac=0.05)
    rng = np.random.default_rng(rdlen)
    for r in reads[:25]:
        r[rng.integers(0, len(r))] = 4                       # Ns in reads
    probs, meta = _problems(synth_genome, reads, truth, sc, rng)
    nfound, naln, ngap = _check(gpu, R, synth_genome, reads, quals, probs, meta)
    assert nfound > 100 and naln > 100
    if indel > 0:
        assert ngap > 0


@pytest.mark.skipif(not have_reference(), reason="oracle/_ref not built")
@pytest.mark.parametrize("mode", ["0", "1", "3"])
def test_dp_e2e_kernel_generations(synth_index, synth_genome, mode):
    """Each end-to-end DP kernel generation (move codes 32-bit, move codes s16x2, H bytes in fill + tail) is the one that
    runs when bt2g_set_dp_mode caps at it, and matches the reference: the first two are the fallbacks when a batch does not
    fit the H-byte kernels."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from torch.profiler import ProfilerActivity, profile
    from bowtie2_b200 import Bt2Gpu
    g = Bt2Gpu(0)
    g.set_dp_mode(int(mode))
    g.load_index_files(synth_index)
    g.set_scoring(local=False)
    R = Reference(synth_index)
    sc = policy.Scoring.default(False)
    reads, quals, truth = synth.make_reads(synth_genome, 120, 100, seed=900 + int(mode), sub_rate=0.02, indel_rate=0.004)
    probs, meta = _problems(synth_genome, reads, truth, sc, np.random.default_rng(5))
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        nfound, naln, ngap = _check(g, R, synth_genome, reads, quals, probs, meta)
    launched = {m.group(1) for e in prof.events() for m in [re.search(r"\b(k_dp_\w+)<", e.name)] if m}
    want = {"0": {"k_dp_e2e"}, "1": {"k_dp_e2e_x2"}, "3": {"k_dp_fill_h", "k_dp_tail_h"}}[mode]
    assert launched == want, launched
    assert nfound > 80 and ngap > 3
    g.close()


@pytest.mark.skipif(not have_reference(), reason="oracle/_ref not built")
def test_dp_e2e_edges(gpu, synth_index, synth_genome):
    """Windows hanging off either reference end, spanning the N gap, repeats (many candidates),
    and a tightened minimum score."""
    gpu.load_index_files(synth_index)
    gpu.set_scoring(local=False)
    R = Reference(synth_index)
    sc = policy.Scoring.default(False)
    g = synth_genome
    rng = np.random.default_rng(3)
    reads, quals, truth = [], [], []
    L = 100
    glen = len(g[0])
    for p in [0, 1, 5, 29, 31, glen - L, glen - L - 1, glen - L - 31, glen // 2 - 60, glen // 2 - 20, glen // 2 + 10]:
        for strand in (1, -1):
            r = g[1][p:p + L].copy()
            r[r > 3] = 0
            r[rng.integers(0, L)] ^= 1
            reads.append(r if strand > 0 else synth.revcomp(r))
            quals.append(rng.integers(35, 74, L).astype(np.uint8))
            truth.append((1, p, strand))
    probs, meta = _problems(g, reads, truth, sc, rng)
    _check(gpu, R, g, reads, quals, probs, meta)
    probs, meta = _problems(g, reads, truth, sc, rng, minsc_bump=40)
    _check(gpu, R, g, reads, quals, probs, meta)


@pytest.mark.skipif(not have_reference(), reason="oracle/_ref not built")
@pytest.mark.parametrize("rdlen,sub,indel", [(100, 0.02, 0.003), (150, 0.03, 0.005), (300, 0.02, 0.004), (60, 0.02, 0.0)])
def test_dp_local_matches_reference(gpu, synth_index, synth_genome, rdlen, sub, indel):
    """--local: floors at 0, candidates anywhere in the rectangle, soft trimming, domination filter."""
    gpu.load_index_files(synth_index)
    gpu.set_scoring(local=True)
    R = Reference(synth_index)
    sc = policy.Scoring.default(True)
    reads, quals, truth = synth.make_reads(synth_genome, 160, rdlen, seed=7 * rdlen, sub_rate=sub, indel_rate=indel, random_frac=0.05)
    rng = np.random.default_rng(rdlen + 1)
    for i, r in enumerate(reads):
        if i % 3 == 0:                                   # junk ends -> soft clipping
            k = int(rng.integers(3, max(4, rdlen // 5)))
            r[:k] = rng.integers(0, 4, k)
        if i % 4 == 0:
            k = int(rng.integers(3, max(4, rdlen // 5)))
            r[-k:] = rng.integers(0, 4, k)
        if i % 11 == 0:
            r[rng.integers(0, rdlen)] = 4
    probs, meta = _problems(synth_genome, reads, truth, sc, rng)
    nfound, naln, ngap = _check(gpu, R, synth_genome, reads, quals, probs, meta, local=True)
    assert nfound > 100 and naln > 100
    gpu.set_scoring(local=False)
