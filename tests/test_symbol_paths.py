"""The base / quality path against plain numpy, exactly, at realistic sizes: the Pass-1 histograms (k_pair_hist_pipe,
k_pair_hist_long, the generic k_pair_hist), the packer (k_pack_tiles, k_pack_long, k_pack_rows) and the decoder
(k_decode_tiles, k_decode_write) at every bit width, every read length residue and every branch a file can take.

Each of these kernel families picks its branch from the shape of the input, and a branch that silently reroutes would
make a test vacuous: every case that targets a branch asserts from the launch timers which kernels ran.

np_pass1 (the reference of the histograms) is itself pinned to the contract emulation (tests/emu.py) on the golden
files by an unmarked test, so it runs without a GPU."""
import types

import numpy as np
import pytest

from conftest import golden_case, load_manifest
from emu import emu_stats

gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------
# numpy reference of Pass 1 (base / quality fields)
# ------------------------------------------------------------------------------------------------
def _ragged_index(starts, lens):
    """flat indices of the segments [starts[i], starts[i] + lens[i])"""
    lens = np.asarray(lens, dtype=np.int64)
    excl = np.cumsum(lens) - lens
    return np.repeat(np.asarray(starts, dtype=np.int64) - excl, lens) + np.arange(int(lens.sum()), dtype=np.int64)


def _record_chunks(lens, budget=1 << 25):
    """[r0, r1) record ranges whose summed lens stay near `budget` (bounds the index arrays of huge files)"""
    c = np.cumsum(np.asarray(lens, dtype=np.int64))
    r0, n = 0, len(c)
    while r0 < n:
        base = c[r0 - 1] if r0 else 0
        r1 = max(int(np.searchsorted(c, base + budget, side="right")), r0 + 1)
        yield r0, min(r1, n)
        r0 = r1


def _lines(a):
    """line geometry of the complete records of a FASTQ (uint8 array) -> (starts, ends) of the four lines, each [n]"""
    nl = np.flatnonzero(a == 10)
    n = len(nl) // 4
    nl = nl[:4 * n].astype(np.int64)
    starts = np.empty(4 * n, dtype=np.int64)
    if n:
        starts[0] = 0
        starts[1:] = nl[:-1] + 1
    return [starts[k::4] for k in range(4)], [nl[k::4] for k in range(4)]


def np_pass1(fastq):
    """The base / quality fields of uqb_analyze from line offsets and bincounts: base_count, qual_count,
    base_single_qual (-1 absent, the quality byte if the base carries exactly one, 256 otherwise), dna_min, dna_max,
    bad_plus_record, bad_len_record.  Bases and qualities pair up position by position over min(len(DNA), len(QUAL)),
    as in the reference's zip."""
    a = np.frombuffer(fastq, dtype=np.uint8)
    (_, d0, p0, q0), (_, d1, _, q1) = _lines(a)
    n = len(d0)
    dlen, qlen = d1 - d0, q1 - q0
    m = np.minimum(dlen, qlen)
    joint = np.zeros(65536, dtype=np.int64)
    for r0, r1 in _record_chunks(m):
        b = a[_ragged_index(d0[r0:r1], m[r0:r1])].astype(np.int32)
        q = a[_ragged_index(q0[r0:r1], m[r0:r1])]
        joint += np.bincount(b * 256 + q, minlength=65536)
    J = joint.reshape(256, 256)
    seen = J > 0
    k = seen.sum(axis=1)
    single = np.where(k == 0, -1, np.where(k == 1, np.argmax(seen, axis=1), 256))
    bad_plus = np.flatnonzero(a[p0] != ord("+")) if n else np.zeros(0, np.int64)     # an empty line 3 reads its '\n'
    bad_len = np.flatnonzero(dlen != qlen)
    return types.SimpleNamespace(
        base_count=J.sum(axis=1).astype(np.uint64), qual_count=J.sum(axis=0).astype(np.uint64),
        base_single_qual=single.astype(np.int64),
        dna_min=int(dlen.min()) if n else 0, dna_max=int(dlen.max()) if n else 0,
        bad_plus_record=int(bad_plus[0]) if bad_plus.size else -1,
        bad_len_record=int(bad_len[0]) if bad_len.size else -1, n_reads=n)


PASS1_ARRAYS = ("base_count", "qual_count", "base_single_qual")
PASS1_SCALARS = ("dna_min", "dna_max", "bad_plus_record", "bad_len_record")


def assert_pass1_equal(got, want, context=""):
    for f in PASS1_SCALARS:
        assert int(getattr(got, f)) == int(getattr(want, f)), "%s %s: %r vs %r" % (context, f, getattr(got, f), getattr(want, f))
    for f in PASS1_ARRAYS:
        g = np.array(list(getattr(got, f)), dtype=np.int64)
        w = np.asarray(getattr(want, f), dtype=np.int64)
        bad = np.flatnonzero(g != w)
        assert bad.size == 0, "%s %s differs at bytes %s: got %s want %s" % (
            context, f, bad[:8].tolist(), g[bad[:8]].tolist(), w[bad[:8]].tolist())


# ------------------------------------------------------------------------------------------------
# FASTQ generator (numpy, no per-record loop)
# ------------------------------------------------------------------------------------------------
def _draw(rng, alphabet, size, weights=None):
    """`size` bytes of `alphabet`; weights (optional, one per symbol) are quantised to 1/256 through a lookup table"""
    sym = np.frombuffer(alphabet.encode("latin-1"), dtype=np.uint8)
    if weights is None:
        return sym[rng.integers(0, len(sym), size=size)]
    w = np.asarray(weights, dtype=np.float64)
    counts = np.maximum(np.round(w / w.sum() * 256).astype(np.int64), 1)
    counts[np.argmax(counts)] -= counts.sum() - 256
    return np.repeat(sym, counts)[rng.integers(0, 256, size=size, dtype=np.uint8)]


def _names(n, long_names=None):
    """QNAME lines '@<lane A-D>:<10000000 + i>' (two columns behind the prefix '@'), or, for the records of
    long_names = (first, count, width), '@rrr...r:<number>' of `width` bytes -> (flat bytes, lengths)"""
    digits = ((10_000_000 + np.arange(n, dtype=np.int64))[:, None] // 10 ** np.arange(7, -1, -1)) % 10 + 48
    short = np.empty((n, 11), dtype=np.uint8)
    short[:, 0] = ord("@")
    short[:, 1] = np.frombuffer(b"ABCD", dtype=np.uint8)[np.arange(n) % 4]
    short[:, 2] = ord(":")
    short[:, 3:] = digits
    lens = np.full(n, 11, dtype=np.int64)
    if long_names is None:
        return short.reshape(-1), lens
    first, count, width = long_names
    lng = np.empty((count, width), dtype=np.uint8)
    lng[:, 0] = ord("@")
    lng[:, 1:width - 9] = ord("r")
    lng[:, width - 9] = ord(":")
    lng[:, width - 8:] = digits[first:first + count]
    lens[first:first + count] = width
    flat = np.concatenate([short[:first].reshape(-1), lng.reshape(-1), short[first + count:].reshape(-1)])
    return flat, lens


def make_fastq(n, length, bases="ACGT", quals="ABCDEFGHIJ", seed=0, base_w=None, qual_w=None, tie=None, plant=(),
               long_names=None):
    """n records; length: an int (fixed-length file) or an int array of n read lengths.
    tie: {base: quality} - every occurrence of the base carries that quality.
    plant: (record, position, base or None, quality or None) - symbols put at given places (after `tie`).
    long_names: (first record, count, width) - a run of records with QNAME lines of `width` bytes."""
    rng = np.random.default_rng(seed)
    lens = np.full(n, int(length), dtype=np.int64) if np.isscalar(length) else np.asarray(length, dtype=np.int64)
    total = int(lens.sum())
    dna = _draw(rng, bases, total, base_w)
    qual = _draw(rng, quals, total, qual_w)
    for b, q in (tie or {}).items():
        qual[dna == ord(b)] = ord(q)
    seq0 = np.cumsum(lens) - lens
    for r, p, b, q in plant:
        assert 0 <= p < lens[r]
        if b is not None:
            dna[seq0[r] + p] = ord(b)
        if q is not None:
            qual[seq0[r] + p] = ord(q)
    names, nlen = _names(n, long_names)
    if long_names is None and np.all(lens == lens[0]):
        L = int(lens[0])
        out = np.empty((n, 11 + 2 * L + 5), dtype=np.uint8)
        out[:, :11] = names.reshape(n, 11)
        out[:, 11] = 10
        out[:, 12:12 + L] = dna.reshape(n, L)
        out[:, 12 + L:15 + L] = np.frombuffer(b"\n+\n", dtype=np.uint8)
        out[:, 15 + L:15 + 2 * L] = qual.reshape(n, L)
        out[:, 15 + 2 * L] = 10
        return out.tobytes()
    rec = nlen + 2 * lens + 5
    st = np.cumsum(rec) - rec
    out = np.full(int(rec.sum()), 10, dtype=np.uint8)
    out[st + nlen + lens + 2] = ord("+")
    name0 = np.cumsum(nlen) - nlen
    for r0, r1 in _record_chunks(nlen + lens):
        out[_ragged_index(st[r0:r1], nlen[r0:r1])] = names[_ragged_index(name0[r0:r1], nlen[r0:r1])]
        src = _ragged_index(seq0[r0:r1], lens[r0:r1])
        out[_ragged_index(st[r0:r1] + nlen[r0:r1] + 1, lens[r0:r1])] = dna[src]
        out[_ragged_index(st[r0:r1] + nlen[r0:r1] + lens[r0:r1] + 4, lens[r0:r1])] = qual[src]
    return out.tobytes()


# ------------------------------------------------------------------------------------------------
# packed tables of the reference
# ------------------------------------------------------------------------------------------------
def ref_tables(fastq, dec):
    """(DNA, QUAL) packed tables of the decision `dec` (host.decide_alphabets): oracle.uq_vec for fixed-length files;
    variable-length rows are the marker (code 1) and the read's symbols, right aligned in rows of dna_max + 1 symbols"""
    from oracle import uq_vec
    if not dec["variable_read_lengths"]:
        _, dna, qual = uq_vec.parse_fixed(fastq, dec["dna_max"])
        return uq_vec.pack_tables(dna, qual, dec)
    a = np.frombuffer(fastq, dtype=np.uint8)
    (_, d0, _, q0), (_, d1, _, _) = _lines(a)
    n, lens = len(d0), d1 - d0
    M = dec["dna_max"] + 1
    base_code = np.zeros(256, dtype=np.uint8)
    qual_code = np.zeros(256, dtype=np.uint8)
    for i, ch in enumerate(dec["bases"]): base_code[ord(ch)] = i
    for i, ch in enumerate(dec["qualities"]): qual_code[ord(ch)] = i
    b = a[_ragged_index(d0, lens)]
    q = a[_ragged_index(q0, lens)]
    cb, cq = base_code[b], qual_code[q]
    for base, code in dec["N_qual"].items():
        t = b == ord(base)
        cb[t] = 0
        cq[t] = code
    rows = np.repeat(np.arange(n), lens)
    cols = _ragged_index(M - lens, lens)
    cd = np.zeros((n, M), dtype=np.uint8)
    cqq = np.zeros((n, M), dtype=np.uint8)
    cd[rows, cols] = cb
    cqq[rows, cols] = cq
    cd[np.arange(n), M - lens - 1] = 1
    cqq[np.arange(n), M - lens - 1] = 1
    return (uq_vec.pack_codes(cd, dec["bits_per_base"], dec["dna_bytes"]),
            uq_vec.pack_codes(cqq, dec["bits_per_quality"], dec["qual_bytes"]))


def assert_table_equal(got, want, name):
    assert got.shape == want.shape, "%s shape %s vs %s" % (name, got.shape, want.shape)
    bad = np.argwhere(got != want)
    assert len(bad) == 0, "%s: %d bytes differ, first at (row, byte) %s" % (name, len(bad), bad[:4].tolist())


def assert_text_equal(got, want):
    if got != want:
        g, w = np.frombuffer(got, np.uint8), np.frombuffer(want, np.uint8)
        k = min(len(g), len(w))
        i = int(np.argmax(g[:k] != w[:k])) if np.any(g[:k] != w[:k]) else k
        raise AssertionError("decoded text differs from the input at byte %d (of %d / %d): got %r want %r" % (
            i, len(g), len(w), got[max(i - 20, 0):i + 20], want[max(i - 20, 0):i + 20]))


# ------------------------------------------------------------------------------------------------
# CPU: the references themselves
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(load_manifest()))
def test_np_pass1_equals_contract_emulation(name):
    fq, _, _ = golden_case(name)
    want, n = emu_stats(fq)
    got = np_pass1(fq)
    assert got.n_reads == n
    assert_pass1_equal(got, want, name)


def test_np_pass1_reports_malformed_records():
    good = b"@r:1\nACGT\n+\nIIII\n"
    st = np_pass1(good + b"@r:2\nACGT\n\nIIII\n" + good + b"@r:3\nACGTA\n+\nIIII\n" + b"@r:4\nAC")
    assert (st.bad_plus_record, st.bad_len_record, st.n_reads) == (1, 3, 4)
    assert (st.dna_min, st.dna_max) == (4, 5)
    assert st.base_count[ord("A")] == 4 and st.qual_count[ord("I")] == 16      # record 3 pairs its first four bases only


def test_generator_and_variable_reference_equal_the_literal_oracle():
    """make_fastq with plants, ties and a long-name run, and ref_tables of a variable-length file, against
    oracle.uq_literal (pinned to the reference-written containers)"""
    from oracle import uq_literal as lit
    from uq_b200 import host
    rng = np.random.default_rng(3)
    fq = make_fastq(700, rng.integers(1, 90, size=700), bases="ACGTN", quals="ABCDEFGHIJ", seed=4, tie={"N": "#"},
                    plant=[(5, 0, "X", "~")], long_names=(300, 150, 60))
    recs = fq.split(b"\n")
    assert recs[4 * 5 + 1][:1] == b"X" and recs[4 * 5 + 3][:1] == b"~" and len(recs[4 * 300]) == 60
    want = {}
    lit.encode(fq, stages=want, sort="None", raw=["DNA", "QUAL", "QNAME"])
    st = np_pass1(fq)
    dec = host.decide_alphabets(st)
    assert dec["bases"] == want["dec"]["bases"] and dec["N_qual"] == want["dec"]["N_qual"] == {"N": 0, "X": 11}
    dna, qual = ref_tables(fq, dec)
    assert_table_equal(dna, want["dna"], "DNA")
    assert_table_equal(qual, want["qual"], "QUAL")


# ------------------------------------------------------------------------------------------------
# the pack / decode grid
# ------------------------------------------------------------------------------------------------
BASE_ALPHABETS = {1: "A", 4: "ACGT", 5: "ACGTN", 9: "ACGTNRYSW", 17: "ACGTNRYSWKMBDHVac"}


def qual_alphabet(k):
    return "".join(chr(33 + i) for i in range(k))


# quality alphabet sizes 2, 5, 9, 17, 33, 65 (2 .. 7 bits) and, with --pad, 5 and 17 (4 and 8 bits); base alphabet sizes
# 1, 4, 5, 9, 17 (2, 2, 3, 4, 5 bits; with --pad 2, 2, 4, 4, 8); read lengths that cover every residue class of a
# 16-symbol chunk that matters (0, 1, 6, 7, 10, 15) and every wd % 4
LENGTHS = [1, 15, 16, 17, 33, 63, 64, 65, 150, 151, 250]
QUAL_SIZES = [(2, False), (5, False), (9, False), (17, False), (33, False), (65, False), (5, True), (17, True)]
BASE_SIZES = [1, 4, 5, 9, 17]
GRID = [(BASE_SIZES[(i + 2 * j) % 5], nq, LENGTHS[(5 * i + j) % 11], pad)
        for i, (nq, pad) in enumerate(QUAL_SIZES) for j in range(5)] + [(17, 17, 64, True), (17, 5, 150, True)]


def test_grid_meets_every_bit_width_at_three_residues():
    from uq_b200 import host
    seen = {}
    for nb, nq, L, pad in GRID:
        seen.setdefault(("DNA", host.bits_for(nb, pad)), set()).add(L % 16)
        seen.setdefault(("QUAL", host.bits_for(nq, pad)), set()).add(L % 16)
    assert {w for t, w in seen if t == "QUAL"} == {2, 3, 4, 5, 6, 7, 8}
    assert {w for t, w in seen if t == "DNA"} == {2, 3, 4, 5, 8}
    thin = {k: sorted(v) for k, v in seen.items() if len(v) < 3}
    assert not thin, thin


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    from uq_b200.device import Context
    c = Context(0)
    c.timing(True)
    yield c
    c.close()


def assert_kernels(report, ran=(), absent=(), what=""):
    names = sorted(report)
    for k in ran:
        assert report.get(k, (0,))[0] > 0, "%s: %s did not run (launched: %s)" % (what, k, names)
    for k in absent:
        assert k not in report, "%s: %s ran (launched: %s)" % (what, k, names)


def analyze(ctx, data, ran=(), absent=(), chunk_bytes=None):
    """device Pass 1 of `data`, compared with np_pass1 field by field -> (device stats, reference stats)"""
    ctx.timing_reset()
    pin = None
    if chunk_bytes is None:
        d = ctx.load_fastq(data)
    else:
        pin = ctx.pinned_empty(len(data))
        pin.array[:] = np.frombuffer(data, dtype=np.uint8)
        d = ctx.load_fastq_streamed(pin, chunk_bytes=chunk_bytes)
    d.split()
    got = d.analyze()
    report = ctx.timing_report()
    d.free()
    if pin is not None:
        pin.free()
    want = np_pass1(data)
    assert_pass1_equal(got, want)
    assert_kernels(report, ran, absent, "analyze")
    return got, want


TILES, LONG, GENERIC = "k_pair_hist_pipe", "k_pair_hist_long", "k_pair_hist"
BENCH_QUALS = "".join(chr(c) for c in range(35, 75))          # '#' .. 'J': about 40 symbols


@pytest.fixture(scope="module")
def bench_like():
    """2 M reads of 150 bp, ACGT with 1 % N, 40 quality symbols"""
    return make_fastq(2_000_000, 150, bases="ACGTN", base_w=[99, 99, 99, 99, 4], quals=BENCH_QUALS, seed=1)


@gpu
def test_hist_bench_like(ctx, bench_like):
    analyze(ctx, bench_like, ran=[TILES], absent=[GENERIC, LONG])


@gpu
@pytest.mark.parametrize("chunk", [1 << 20, 48 << 10])
def test_hist_streamed_chunks_start_inside_tiles(ctx, bench_like, chunk):
    """chunks of the streamed load end in the middle of a record tile: the tile kernel runs on ranges that start anywhere"""
    analyze(ctx, bench_like, ran=[TILES], absent=[GENERIC, LONG], chunk_bytes=chunk)


@gpu
@pytest.mark.parametrize("kind", ["one_quality", "novaseq", "longest_tile", "short_then_long", "soft_masked"])
def test_hist_multi_tile(ctx, kind):
    """1 M reads, 50 - 60 tiles per CTA: the three-stage buffer rotation, the hints a CTA learns from its first tile, the
    adaptive meetings of the 8-bit quality columns and the offender flush"""
    n = 1_000_003
    if kind == "one_quality":            # every base carries 'I': no base ever becomes a hint, the busiest column fills fastest
        data = make_fastq(n, 150, bases="ACGTN", base_w=[60, 60, 60, 60, 16], quals="I", seed=2)
    elif kind == "novaseq":              # four binned quality symbols
        data = make_fastq(n, 151, quals="#,:F", qual_w=[2, 5, 20, 73], seed=3)
    elif kind == "longest_tile":         # 382-byte records: 128 of them just fit a 48 KB tile
        data = make_fastq(n, 183, bases="ACGTN", base_w=[60, 60, 60, 60, 16], quals=BENCH_QUALS, seed=4)
    elif kind == "short_then_long":
        # 20 bp reads space the meetings of the CTA 13 tiles apart; from tile 27 of every CTA on (148 CTAs) the reads are
        # 183 bp long, and a quality thread meets some 800 symbols - mostly 'F' - before the next meeting: only the
        # thread-private column flush keeps its 8-bit counters from wrapping
        lens = np.where(np.arange(n) < 148 * 27 * 128, 20, 183)
        data = make_fastq(n, lens, quals="#,:F", qual_w=[2, 5, 20, 73], seed=5)
    else:                                # half of the bases are offenders of the four hints, which keep changing
        data = make_fastq(n, 150, bases="acgtACGTRYSWKMBDHVN", base_w=[60] * 8 + [1] * 11, quals=BENCH_QUALS, seed=6)
    got, want = analyze(ctx, data, ran=[TILES], absent=[GENERIC, LONG])
    if kind == "one_quality":
        assert all(want.base_single_qual[ord(b)] == ord("I") for b in "ACGTN")
    if kind == "short_then_long":
        assert (want.dna_min, want.dna_max) == (20, 183)


# record index of tile 40 of CTA 3 (148 CTAs, one per SM): deep in a CTA's tiles, long after its hints were learnt
DEEP = (148 * 40 + 3) * 128 + 7
RARE_N = 1_000_037                        # the last tile holds 37 records


@gpu
def test_hist_rare_symbols_at_edges(ctx):
    """quality and base bytes that occur exactly once, each at another edge: first and last byte of the file, both sides of
    the 16-byte unit and 64-byte boundaries, both sides of a tile boundary, the partial last tile, deep in a CTA's tiles;
    '!' (33) and '~' (126) are the ends of the tile kernel's quality range"""
    L = 150
    places = [(0, 0), (RARE_N - 1, L - 1), (500, 15), (501, 16), (502, 63), (503, 64), (127, L - 1), (128, 0),
              (RARE_N - 20, 77), (DEEP, 31)]
    rare_q = "!~\"}$|%{&'"
    rare_b = "XZBDHV*xzb"
    plant = [(r, p, b, q) for (r, p), b, q in zip(places, rare_b, rare_q)]
    data = make_fastq(RARE_N, L, bases="ACGTN", base_w=[60, 60, 60, 60, 16], quals="".join(chr(c) for c in range(40, 81)),
                      seed=7, plant=plant)
    got, want = analyze(ctx, data, ran=[TILES], absent=[GENERIC, LONG])
    for b, q in zip(rare_b, rare_q):
        assert want.base_count[ord(b)] == 1 and want.qual_count[ord(q)] == 1
        assert want.base_single_qual[ord(b)] == ord(q)


@gpu
@pytest.mark.parametrize("other", [False, True])
def test_hist_single_quality_state(ctx, other):
    """N always carries '#' - except, in one variant, once near the end of the file"""
    n = 1_000_003
    plant = [(n - 5_000, 42, "N", "B")] if other else []
    data = make_fastq(n, 150, bases="ACGTN", base_w=[60, 60, 60, 60, 16], seed=8, tie={"N": "#"}, plant=plant)
    got, want = analyze(ctx, data, ran=[TILES], absent=[GENERIC, LONG])
    assert want.base_single_qual[ord("N")] == (256 if other else ord("#"))


@gpu
@pytest.mark.parametrize("shared", [False, True])
def test_hist_ntrick_decision_on_exact_counts(ctx, shared):
    """'#' belongs to N alone (N_qual = its index in the qualities) - or one 'A' at a tile edge carries it, too, and the
    decision takes the "new quality" branch (N_qual = len(qualities) + 1)"""
    from uq_b200 import host
    n = 1_000_003
    plant = [(128, 0, "A", "#")] if shared else []
    data = make_fastq(n, 150, bases="ACGTN", base_w=[60, 60, 60, 60, 16], seed=9, tie={"N": "#"}, plant=plant)
    got, want = analyze(ctx, data, ran=[TILES], absent=[GENERIC, LONG])
    dec_g, dec_w = host.decide_alphabets(got), host.decide_alphabets(want)
    assert dec_g == dec_w
    quals = dec_w["qualities"]
    assert dec_w["N_qual"] == ({"N": len(quals) + 1} if shared else {"N": quals.index("#")})


@gpu
@pytest.mark.parametrize("q", [32, 127, 200])
def test_hist_quality_outside_the_tile_range_takes_the_generic_kernel(ctx, q):
    n = 300_001
    data = bytearray(make_fastq(n, 150, quals=BENCH_QUALS, seed=10))
    data[data.index(b"#", len(data) * 2 // 3)] = q                    # '#' occurs in quality lines only
    analyze(ctx, bytes(data), ran=[TILES, GENERIC], absent=[LONG])


@gpu
@pytest.mark.parametrize("kind", ["fixed_2kb", "variable_1_20kb"])
def test_hist_long_reads(ctx, kind):
    n = 20_000
    if kind == "fixed_2kb":
        data = make_fastq(n, 2_000, bases="ACGTN", base_w=[60, 60, 60, 60, 16], quals=BENCH_QUALS, seed=11,
                          plant=[(n - 1, 1_999, "X", "~"), (7, 0, "Z", "!")])
    else:
        lens = np.random.default_rng(12).integers(1_000, 20_001, size=n)
        data = make_fastq(n, lens, bases="ACGTN", base_w=[60, 60, 60, 60, 16], quals=BENCH_QUALS, seed=12, tie={"N": "#"})
    analyze(ctx, data, ran=[LONG], absent=[GENERIC, TILES])


LONG_NAME_RUN = (400_003, 300, 200)


@gpu
def test_hist_tile_that_does_not_fit(ctx):
    """a run of 300 records with 200-byte names in a file whose mean record fits: the tiles of the run exceed 48 KB, the
    tile kernel gives up mid-kernel and the generic kernel recounts the file"""
    data = make_fastq(1_000_003, 150, bases="ACGTN", base_w=[60, 60, 60, 60, 16], quals=BENCH_QUALS, seed=13,
                      long_names=LONG_NAME_RUN)
    assert len(data) // 1_000_003 <= 383
    analyze(ctx, data, ran=[TILES, GENERIC], absent=[LONG])


# ---- pack and decode --------------------------------------------------------------------------
def pack_decode(ctx, data, pad=False, pack_ran=(), pack_absent=(), decode_ran=(), decode_absent=(), keyed=True):
    """host.encode_device on `data`: the decision equals host.decide_alphabets of np_pass1, the packed tables equal
    ref_tables byte for byte, the raw container decodes to `data` byte for byte; keyed (sort DNA / QUAL): the unique
    tables and keys equal numpy's stable sort / unique of the reference tables.  -> the decision"""
    from oracle import uq_vec
    from uq_b200 import host
    dec_w = host.decide_alphabets(np_pass1(data), pad=pad)
    dna_w, qual_w = ref_tables(data, dec_w)
    fq = ctx.load_fastq(data)
    st = {}
    ctx.timing_reset()
    members, cfg = host.encode_device(ctx, fq, sort="None", raw=["DNA", "QUAL", "QNAME"], pad=pad, stages=st)
    assert_kernels(ctx.timing_report(), pack_ran, pack_absent, "pack")
    assert st["dec"] == dec_w
    assert_table_equal(st["dna"].download().reshape(dna_w.shape), dna_w, "DNA")
    assert_table_equal(st["qual"].download().reshape(qual_w.shape), qual_w, "QUAL")
    host_members = members.download()
    members.free()
    for a in [st["dna"], st["qual"]] + st["cols"]:
        a.free()
    fq.free()
    ctx.timing_reset()
    out = host.decode(host_members, cfg, ctx=ctx).tobytes()
    assert_kernels(ctx.timing_report(), decode_ran, decode_absent, "decode")
    assert_text_equal(out, data)
    if keyed:
        ref = {"DNA": uq_vec.sort_unique(dna_w), "QUAL": uq_vec.sort_unique(qual_w)}
        for sort, other in (("DNA", "QUAL"), ("QUAL", "DNA")):
            fq = ctx.load_fastq(data)
            members, _ = host.encode_device(ctx, fq, sort=sort, pad=pad)
            got = members.download()
            members.free()
            fq.free()
            perm = ref[sort][0]
            for t in (sort, other):
                _, key, uniq = ref[t]
                assert_table_equal(got[t], uniq, "sort=%s unique %s" % (sort, t))
                assert np.array_equal(got[t + ".key"].astype(np.int64), key[perm]), "sort=%s %s.key" % (sort, t)
    return dec_w


TILE_REC_MAX = 383       # mean (and per-tile) record bytes of the tile paths of the histogram and the packer
DECODE_REC_MAX = 431     # mean record bytes of the tiled decoder


@gpu
@pytest.mark.parametrize("nb,nq,L,pad", GRID)
def test_pack_decode_fixed_length_grid(ctx, nb, nq, L, pad):
    """every bit width of both tables at three or more residues of L mod 16; 1 000 reads are seven full 128-record
    tiles (fifteen 64-record decode tiles) and a partial one"""
    from uq_b200 import host
    n = 1_000
    data = make_fastq(n, L, bases=BASE_ALPHABETS[nb], quals=qual_alphabet(nq), seed=100 + 7 * L + nb + nq)
    rec = len(data) // n
    if rec <= TILE_REC_MAX:
        pack_ran, pack_absent = ["k_pack_tiles"], ["k_pack_long", "k_pack_rows"]
    else:
        pack_ran, pack_absent = ["k_pack_long"], ["k_pack_tiles", "k_pack_rows"]
    dec_ran, dec_absent = (["k_decode_tiles"], ["k_decode_write"]) if rec <= DECODE_REC_MAX else (["k_decode_write"], ["k_decode_tiles"])
    dec = pack_decode(ctx, data, pad, pack_ran, pack_absent, dec_ran, dec_absent)
    assert (dec["bits_per_base"], dec["bits_per_quality"]) == (host.bits_for(nb, pad), host.bits_for(nq, pad))
    assert dec["N_qual"] == {} and not dec["variable_read_lengths"]


VARIABLE = [(4, 33, 1, 50, False), (5, 9, 20, 63, False), (17, 2, 1, 63, False),
            (4, 65, 30, 151, False), (17, 17, 1, 250, False), (5, 17, 60, 120, True), (9, 5, 64, 64 + 15, False)]


@gpu
@pytest.mark.parametrize("nb,nq,lo,hi,pad", VARIABLE)
def test_pack_decode_variable_length(ctx, nb, nq, lo, hi, pad):
    """variable-length rows (marker + symbols, right aligned): the one-warp-per-read packer below 64 bases, the
    one-CTA-per-read packer from 64 on; the decoder writes them one warp per read"""
    n = 1_000
    lens = np.random.default_rng(lo + hi).integers(lo, hi + 1, size=n)
    lens[0], lens[-1] = lo, hi
    data = make_fastq(n, lens, bases=BASE_ALPHABETS[nb], quals=qual_alphabet(nq), seed=200 + hi + nb + nq)
    packer = "k_pack_long" if hi >= 64 else "k_pack_rows"
    other = "k_pack_rows" if packer == "k_pack_long" else "k_pack_long"
    dec = pack_decode(ctx, data, pad, [packer], ["k_pack_tiles", other], ["k_decode_write"], ["k_decode_tiles"])
    assert dec["variable_read_lengths"] and dec["dna_max"] == hi


@gpu
def test_pack_decode_tile_that_does_not_fit(ctx):
    """the 200-byte-name run inside a fixed-length file: the histogram, the packer and the decoder each give up on the
    tiles of the run mid-kernel and redo the file on their direct-from-global path"""
    n = 5_003
    data = make_fastq(n, 150, bases="ACGTN", base_w=[60, 60, 60, 60, 16], quals=BENCH_QUALS, seed=14,
                      long_names=(2_001, 300, 200))
    assert len(data) // n <= TILE_REC_MAX
    analyze(ctx, data, ran=[TILES, GENERIC])
    pack_decode(ctx, data, pack_ran=["k_pack_tiles", "k_pack_long"], decode_ran=["k_decode_tiles", "k_decode_write"])


@gpu
def test_decode_restoration_list_overflows(ctx):
    """150 bp reads with about 19 tricked N each: a 64-record decode tile holds some 1 200 restorations, more than its
    list of 512; the two-bit DNA writer then walks the quality codes again"""
    data = make_fastq(2_003, 150, bases="ACGTN", base_w=[56, 56, 56, 56, 32], seed=15, tie={"N": "#"})
    a = np.frombuffer(data, np.uint8)
    (_, d0, _, _), _ = _lines(a)
    per_read = np.add.reduceat((a == ord("N")).astype(np.int64), d0)[:64]
    assert per_read.min() >= 10
    dec = pack_decode(ctx, data, pack_ran=["k_pack_tiles"], decode_ran=["k_decode_tiles"], decode_absent=["k_decode_write"])
    assert dec["bits_per_base"] == 2 and dec["N_qual"] == {"N": dec["qualities"].index("#")}


@gpu
@pytest.mark.parametrize("shared", [False, True])
def test_decode_two_tricked_bases(ctx, shared):
    """Q10: two bases with their own single quality, N with '#' and '.' with '!'; shared: 'A' and 'C' carry those
    qualities too, so both take the "new quality" branch and their codes depend on the order the bases are visited"""
    n = 2_003
    plant = [(130, 3, "A", "#"), (1_000, 149, "C", "!")] if shared else []
    data = make_fastq(n, 150, bases="ACGTN.", base_w=[60, 60, 60, 60, 8, 8], quals="ABCDEFGHIJ", seed=16,
                      tie={"N": "#", ".": "!"}, plant=plant)
    dec = pack_decode(ctx, data, pack_ran=["k_pack_tiles"], decode_ran=["k_decode_tiles"], decode_absent=["k_decode_write"])
    q = dec["qualities"]
    if shared:
        assert dec["N_qual"] == {".": len(q) + 1, "N": len(q) + 2}
    else:
        assert dec["N_qual"] == {".": q.index("!"), "N": q.index("#")}
