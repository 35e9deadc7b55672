"""CPU: the torch index builder must reproduce bowtie2-build-s output byte for byte."""
import os

import numpy as np
import pytest
import torch

from bowtie2_b200 import synth
from bowtie2_b200.index_build import build_index, suffix_array
from oracle_lib import build_reference_index


def test_suffix_array_small():
    rng = np.random.default_rng(0)
    for n in (1, 2, 5, 30, 200, 3000):
        for alpha in (1, 2, 4):
            s = rng.integers(0, alpha, n).astype(np.uint8)
            sa, isa = suffix_array(torch.from_numpy(s))
            # brute force with "end of text is largest": compare as tuples padded with 4
            suf = sorted(range(n + 1), key=lambda i: tuple(s[i:]) + (4,))
            assert sa.tolist() == suf, (n, alpha)
            assert isa[sa].tolist() == list(range(n + 1))


def test_index_files_identical_to_bowtie2_build(tmp_path, synth_genome, synth_index):
    contigs = [torch.from_numpy(c) for c in synth_genome]
    ix = build_index(contigs)
    base = str(tmp_path / "mine")
    ix.write_files(base)
    for suf in ("1.bt2", "2.bt2", "3.bt2", "4.bt2", "rev.1.bt2"):
        a = open(f"{base}.{suf}", "rb").read()
        b = open(f"{synth_index}.{suf}", "rb").read()
        assert len(a) == len(b), (suf, len(a), len(b))
        if a != b:
            diff = [i for i in range(len(a)) if a[i] != b[i]]
            raise AssertionError(f"{suf}: {len(diff)} differing bytes, first at {diff[:10]}")


def test_index_with_repeats_and_short_contigs(tmp_path):
    """Long exact repeats (deep prefix doubling), tiny contigs and contig-edge N runs."""
    rng = np.random.default_rng(5)
    unit = rng.integers(0, 4, 700).astype(np.uint8)
    g = [np.concatenate([unit, unit, rng.integers(0, 4, 50).astype(np.uint8), unit]),
         np.concatenate([np.full(7, 4, np.uint8), rng.integers(0, 4, 40).astype(np.uint8), np.full(3, 4, np.uint8),
                         np.zeros(300, np.uint8), np.full(5, 4, np.uint8)]),
         rng.integers(0, 4, 12).astype(np.uint8)]
    fa = str(tmp_path / "g.fa")
    synth.write_fasta(fa, g)
    want = str(tmp_path / "want")
    build_reference_index("bowtie2-build-s", fa, want)
    ix = build_index([torch.from_numpy(c) for c in g])
    base = str(tmp_path / "mine")
    ix.write_files(base)
    for suf in ("1.bt2", "2.bt2", "3.bt2", "4.bt2", "rev.1.bt2"):
        a = open(f"{base}.{suf}", "rb").read()
        b = open(f"{want}.{suf}", "rb").read()
        assert a == b, (suf, len(a), len(b), [i for i in range(min(len(a), len(b))) if a[i] != b[i]][:10])
