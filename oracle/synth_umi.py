"""Synthetic FASTQ kind 'umi' (host / numpy): the 'illumina' records of oracle/synth.py with '_<UMI>' appended to
the header, as UMI extraction tools write it.  The UMI is 6-12 symbols of ACGTN; its length and its symbols come from
their own stream ids, so the DNA and quality lines are exactly those of kind 'illumina'.

TEST INFRASTRUCTURE.  The device generator (uq_b200/csrc/synth.cu, uqb_synth kind 4) produces the same bytes; the
UMI column is a 'strings' QNAME column (declared extension E1, DESIGN section 4).
"""
import numpy as np

from .synth import make_records, rnd

ST_UMI_LEN, ST_UMI = 20, 21      # stream ids shared with synth.cu
ACGTN = np.frombuffer(b"ACGTN", dtype=np.uint8)


def umi_of(seed, r):
    """UMI bytes of record r (global index)"""
    n = 6 + int(rnd(seed, ST_UMI_LEN, r) % np.uint64(7))
    with np.errstate(over="ignore"):
        idx = np.uint64(r) * np.uint64(16) + np.arange(n, dtype=np.uint64)
    return ACGTN[(rnd(seed, ST_UMI, idx) % np.uint64(5)).astype(np.int64)].tobytes()


def make_records_umi(n=1000, length=100, seed=1, first=0):
    recs = make_records(kind="illumina", n=n, length=length, seed=seed, first=first)
    return [(h + b"_" + umi_of(seed, first + i), d, q) for i, (h, d, q) in enumerate(recs)]


def make_fastq_umi(**kw):
    return b"".join(h + b"\n" + d + b"\n+\n" + q + b"\n" for h, d, q in make_records_umi(**kw))
