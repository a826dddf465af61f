"""Synthetic FASTQ kinds 'renamed' and 'mixed' (host / numpy): QNAMEs that do not split into columns.

TEST INFRASTRUCTURE.  The device generator (uq_b200/csrc/synth.cu, uqb_synth kinds 5 and 6) produces the same bytes.
The DNA and quality lines are those of kind 'illumina' of oracle/synth.py; only the header differs:

  renamed : @SRR0000001.<record + 1>, as read renaming tools write it.  No character has a constant count.
  mixed   : blocks of 1024 records alternate between the 'casava' header of oracle/synth.py and the pre-1.8 Illumina
            header @HWI-D00123:<lane>:<tile>:<x>:<y>#0/1, as in a file concatenated from two runs: ':' occurs 9 times
            in one style and 4 times in the other.

Both files are stored as one QNAME column (declared extension E2, DESIGN section 4).
"""
from .synth import make_records

BLOCK = 1024


def make_records_names(kind="renamed", n=1000, length=100, seed=1, first=0):
    if kind == "renamed":
        recs = make_records(kind="illumina", n=n, length=length, seed=seed, first=first)
        return [(b"@SRR0000001.%d" % (first + i + 1), d, q) for i, (_, d, q) in enumerate(recs)]
    if kind != "mixed":
        raise ValueError(kind)
    casava = make_records(kind="casava", n=n, length=length, seed=seed, first=first)
    plain = make_records(kind="illumina", n=n, length=length, seed=seed, first=first)
    out = []
    for i, ((hc, d, q), (hp, _, _)) in enumerate(zip(casava, plain)):
        if (first + i) // BLOCK % 2 == 0:
            out.append((hc, d, q))
        else:                                   # same lane / tile / x / y streams as the other headers
            out.append((b"@HWI-D00123:" + hp[len(b"@SIM001:1:FCX123:"):] + b"#0/1", d, q))
    return out


def make_fastq_names(**kw):
    return b"".join(h + b"\n" + d + b"\n+\n" + q + b"\n" for h, d, q in make_records_names(**kw))
