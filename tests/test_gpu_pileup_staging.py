"""The cases of test_sim_pileup_staging.py on the B200, plus a chr19-length contig of 30x short reads with reads of more
than 1024 CIGAR or mask words mixed in."""
import pytest

from test_sim_pileup_staging import (case_many_chunks, case_nonmonotonic_qual_offsets, case_overflow, case_residues, case_split, case_tile_edges, check,
                                     overflow_reads, short_reads)
from rsicnv_b200 import synth

pytestmark = pytest.mark.gpu


def test_many_chunks(gpu_lib, oracle):
    case_many_chunks(gpu_lib, oracle)


def test_overflow_among_short_reads(gpu_lib, oracle):
    case_overflow(gpu_lib, oracle)


def test_nonmonotonic_qual_offsets(gpu_lib, oracle):
    case_nonmonotonic_qual_offsets(gpu_lib, oracle)


def test_start_residues(gpu_lib, oracle):
    case_residues(gpu_lib, oracle)


def test_tile_edges(gpu_lib, oracle):
    case_tile_edges(gpu_lib, oracle)


@pytest.mark.parametrize("nparts", [2, 3])
def test_split_run(gpu_lib, nparts):
    case_split(gpu_lib, nparts)


def test_chr19_length_with_overflow_reads(gpu_lib, oracle):
    L = synth.CHR19_LEN
    fa, short = short_reads(L, 36)
    check(gpu_lib, oracle, fa, synth.merge_reads(short, overflow_reads(L, 36)), "chr19 length, 30x + reads larger than a stage")
