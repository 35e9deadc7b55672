import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _build_index(builder, fasta, base, extra=()):
    from oracle_lib import build_reference_index
    build_reference_index(builder, fasta, base, extra)


@pytest.fixture(scope="session")
def lambda_index(tmp_path_factory):
    d = tmp_path_factory.mktemp("lambda")
    base = str(d / "lambda")
    _build_index("bowtie2-build-s", os.path.join(GOLDEN, "lambda_virus.fa"), base)
    return base


@pytest.fixture(scope="session")
def rep_index(tmp_path_factory):
    """index of the repeat-rich golden genome (tests/golden/rep_genome.fa: ctg1 14000 bp, ctg2 10000 bp)"""
    d = tmp_path_factory.mktemp("rep")
    base = str(d / "rep")
    _build_index("bowtie2-build-s", os.path.join(GOLDEN, "rep_genome.fa"), base)
    return base


@pytest.fixture(scope="session")
def synth_genome():
    from bowtie2_b200 import synth
    return synth.make_genome(n_contigs=3, contig_len=40000, seed=11, repeat_frac=0.05, repeat_len=300,
                             repeat_copies=12, n_gap=37)


@pytest.fixture(scope="session")
def synth_index(tmp_path_factory, synth_genome):
    """Small .bt2 index over a 3-contig genome with repeats and N gaps (offrate 4 default)."""
    from bowtie2_b200 import synth
    d = tmp_path_factory.mktemp("synth_s")
    fa = str(d / "g.fa")
    synth.write_fasta(fa, synth_genome)
    base = str(d / "g")
    _build_index("bowtie2-build-s", fa, base)
    return base


@pytest.fixture(scope="session")
def synth_index_large(tmp_path_factory, synth_genome):
    """Same genome as a .bt2l (64-bit offsets, 128 B sides) index."""
    from bowtie2_b200 import synth
    d = tmp_path_factory.mktemp("synth_l")
    fa = str(d / "g.fa")
    synth.write_fasta(fa, synth_genome)
    base = str(d / "g")
    _build_index("bowtie2-build-l", fa, base)
    return base


@pytest.fixture(scope="session")
def golden_fm():
    return np.load(os.path.join(GOLDEN, "lambda_fm_golden.npz"))


def read_fastq_codes(path, n):
    code = {"A": 0, "C": 1, "G": 2, "T": 3}
    reads, quals, names = [], [], []
    with open(path) as f:
        for _ in range(n):
            name = f.readline().strip()
            seq = f.readline().strip()
            f.readline()
            q = f.readline().strip()
            if not q:
                break
            names.append(name[1:])
            reads.append(np.array([code.get(c, 4) for c in seq], dtype=np.uint8))
            quals.append(np.frombuffer(q.encode(), dtype=np.uint8).copy())
    return names, reads, quals


@pytest.fixture(scope="session")
def lambda_reads():
    return read_fastq_codes(os.path.join(GOLDEN, "lambda_reads_1.fq"), 2000)


@pytest.fixture(scope="session")
def gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from bowtie2_b200 import Bt2Gpu
    return Bt2Gpu(0)
