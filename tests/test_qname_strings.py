"""'strings' QNAME columns (declared extension E1, DESIGN section 4): a column that leaves 'mapping' and is not all
integers is stored as the tokens themselves, an |S<W> array with W = the longest token.  Host decisions and the
oracle run without a GPU; the device encode, the columns <-> rows transforms with byte columns, the decode, the --test
feed, the sharded path and the CLI are checked on the GPU against the oracle."""
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, assert_config_equal, assert_members_equal, records_multiset

MIXES = [dict(sort=s, raw=r) for s in ("None", "DNA", "QNAME") for r in (None, ["QNAME"])]


# ------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------
def fastq_of(names, length=12, seed=1):
    """header lines (without '@') -> FASTQ bytes with random fixed-length reads"""
    rng = random.Random(seed)
    out = []
    for h in names:
        dna = "".join(rng.choice("ACGT") for _ in range(length))
        qual = "".join(rng.choice("ABCDEFGHIJ") for _ in range(length))
        out.append("@%s\n%s\n+\n%s\n" % (h, dna, qual))
    return "".join(out).encode("latin-1")


def _word(rng, n, alphabet="ACGTN"):
    return "".join(rng.choice(alphabet) for _ in range(n))


def umi_fastq(n, seed=5, length=30):
    from oracle.synth_umi import make_fastq_umi
    return make_fastq_umi(n=n, length=length, seed=seed)


def varlen_names(n=400, seed=2):
    """tokens of length 0 .. 40, and one each of length 0, 1 and 255"""
    rng = random.Random(seed)
    toks = [_word(rng, rng.randrange(0, 41)) for _ in range(n)]
    toks[3], toks[50], toks[200] = "", "G", _word(rng, 255)
    return ["r:%d:%s" % (i, t) for i, t in enumerate(toks)]


def position_names(where, n=300, seed=3):
    rng = random.Random(seed)
    out = []
    for i in range(n):
        tok = _word(rng, rng.randrange(3, 9))
        ints = [str(i), str(rng.randrange(4))]
        cols = {"first": [tok] + ints, "middle": [ints[0], tok, ints[1]], "last": ints + [tok]}[where]
        out.append("p:" + ":".join(cols))
    return out


def two_string_names(n=300, seed=4):
    rng = random.Random(seed)
    return ["t:%s:%d:%s" % (_word(rng, rng.randrange(2, 7)), i, _word(rng, rng.randrange(1, 10), "ACGTNXYZ")) for i in range(n)]


def width_names(w, n=150, seed=6):
    """a string column of exactly w bytes between two integer columns: a byte-order mix-up between string and integer
    columns changes the QNAME order"""
    rng = random.Random(seed + w)
    return ["w:%d:%s:%d" % (rng.randrange(300), _word(rng, w, "ABCDEFGHIJKLMNOPQRSTUVWXYZ"), rng.randrange(3)) for _ in range(n)]


def late_names(n=25100, switch=25000, seed=7):
    """column 2 is integers (8 digits with leading zeros) after checkpoint 0 and turns into strings at record `switch`:
    the longest token (8) is longer than the reference's own `longest` (len(str(max)))"""
    rng = random.Random(seed)
    out = []
    for i in range(n):
        tok = "%08d" % rng.randrange(10 ** 6) if i < switch else "X%d" % rng.randrange(1000)
        out.append("l:%d:%s" % (rng.randrange(4), tok))
    return out


def long_names(n=400, seed=8):
    """later QNAME lines much longer than the first one: no compact QNAME array, the tokens are read from the FASTQ"""
    rng = random.Random(seed)
    return ["f:%d:%s" % (i, _word(rng, 4 if i == 0 else rng.randrange(4, 120))) for i in range(n)]


def sort_key(name, columns, prefix, suffix, seps):
    """E1 order of one record's tokens: mapping as the token text, integers as ints, strings as bytes"""
    import re
    mid = name[len(prefix):len(name) - len(suffix)]
    toks = re.split("(?:%s)" % "|".join(re.escape(s) for s in seps), mid) if seps else [mid]
    key = []
    for t, c in zip(toks, columns):
        if c["format"] == "integers":
            key.append(int(t))
        elif c["format"] == "strings":
            key.append(t.encode("latin-1"))
        else:
            key.append(t)
    return tuple(key)


def _records(fq):
    ls = fq.split(b"\n")[:-1]
    return [tuple(ls[i:i + 4]) for i in range(0, len(ls), 4)]


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def _colstats(all_int, distinct0, max_len, n_reads, n_distinct=None):
    from uq_b200 import _lib as L
    cs = L.ColStats()
    cs.all_int = 1 if all_int else 0
    cs.min_val, cs.max_val = 0, 99
    cs.min_len, cs.max_len = 1, max_len
    ncheck = 0
    t = 10000
    while t <= n_reads - 1:
        ncheck += 1
        t *= 2
    cs.n_checkpoints = ncheck
    cs.distinct_at[0] = distinct0
    for k in range(1, L.MAX_CHECKPOINTS):
        cs.distinct_at[k] = L.U64_MAX
    cs.n_distinct = L.U64_MAX if n_distinct is None else n_distinct
    return cs


def test_decide_columns_strings_integers_and_the_width_limit():
    from uq_b200 import host
    cols = host.decide_columns([_colstats(False, 5000, 12, 30000), _colstats(True, 5000, 2, 30000)], 30000, None)
    assert cols[0] == {"name": "QNAME_1", "format": "strings", "longest": 12, "dtype": "|S12"}
    assert cols[1]["format"] == "integers" and cols[1]["dtype"] == "uint8" and not cols[1]["offset"]
    assert host.column_specs(cols)[0] == (2, 12, False, 0)
    assert host.qname_kinds(cols) == [1, 0]
    assert host.qname_kinds(cols[1:]) is None
    # demoted at the end of a small file
    small = host.decide_columns([_colstats(False, 0, 3, 50, n_distinct=40)], 50, None)
    assert small[0]["dtype"] == "|S3"
    assert host.decide_columns([_colstats(False, 5000, 255, 30000)], 30000, None)[0]["dtype"] == "|S255"
    with pytest.raises(host.UQError, match="QNAME column 1 holds a token of 256 bytes"):
        host.decide_columns([_colstats(False, 5000, 256, 30000)], 30000, None)


def _oracle_round_trip(fq):
    from oracle import uq_strings as lit
    m, c = lit.encode(fq)
    assert lit.decode(m, c) == fq
    cols = c["QNAME_columns"]
    assert any(col["format"] == "strings" for col in cols)
    for mix in MIXES[2:]:
        m, c = lit.encode(fq, **mix)
        text = lit.decode(m, c)
        assert records_multiset(text) == records_multiset(fq)
        if mix["sort"] == "QNAME":
            recs = _records(fq)
            names = [r[0].decode("latin-1") for r in recs]
            args = (cols, c["QNAME_prefix"], c["QNAME_suffix"], c["QNAME_separators"])
            order = sorted(range(len(recs)), key=lambda i: sort_key(names[i], *args))      # stable
            assert _records(text) == [recs[i] for i in order]
    return cols


def test_oracle_round_trip_umi_reads_across_checkpoints():
    cols = _oracle_round_trip(umi_fastq(30000, length=8))
    assert cols[-1]["format"] == "strings" and cols[-1]["dtype"] == "|S12"


def test_oracle_round_trip_variable_length_tokens():
    cols = _oracle_round_trip(fastq_of(varlen_names()))
    assert cols[1] == {"name": "QNAME_2", "format": "strings", "longest": 255, "dtype": "|S255"}


def test_oracle_round_trip_late_integers_to_strings():
    cols = _oracle_round_trip(fastq_of(late_names(), length=6))
    assert cols[1]["format"] == "strings" and cols[1]["longest"] == 8 and cols[1]["dtype"] == "|S8"


@pytest.mark.parametrize("name", ["c2_keyed_sortQNAME", "c3_casava_sortQNAME", "c6_checkpoints", "c7_offset_suffix_keyed"])
def test_strings_oracle_reproduces_reference_containers(name):
    """on files without string columns the E1 oracle is the literal oracle: the reference-written containers"""
    from conftest import golden_case
    from oracle import uq_strings
    from uq_b200 import container
    fq, uq, kw = golden_case(name)
    want, want_cfg = container.read_container(uq)
    got, cfg = uq_strings.encode(fq, **kw)
    assert_members_equal(got, want, name)
    assert_config_equal(cfg, want_cfg, name)
    assert uq_strings.decode(want, want_cfg) == __import__("oracle.uq_literal", fromlist=["decode"]).decode(want, want_cfg)


def test_planned_writer_with_string_members(tmp_path):
    from oracle import uq_strings as lit
    from uq_b200 import container
    fq = fastq_of(two_string_names())
    for mix in (dict(), dict(sort="QNAME", raw=["QNAME"])):
        members, config = lit.encode(fq, **mix)
        assert any(v.dtype.kind == "S" for v in members.values())
        a, b = str(tmp_path / "planned.uQ"), str(tmp_path / "tarfile.uQ")
        plan = container.write_container(a, members, config)
        container.write_container_tarfile(b, members, config)
        da, db = open(a, "rb").read(), open(b, "rb").read()
        assert len(da) == plan.total and da == db
        for mm in (False, True):
            got, cfg = container.read_container(a, mmap=mm)
            assert json.dumps(cfg, sort_keys=True) == json.dumps(json.loads(json.dumps(config)), sort_keys=True)
            for k, v in members.items():
                assert got[k].dtype == v.dtype and np.array_equal(got[k], v), k


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    from uq_b200.device import Context
    c = Context(0)
    yield c
    c.close()


@pytest.mark.gpu
def test_device_synth_umi_matches_host(ctx):
    from oracle import synth
    from oracle.synth_umi import make_fastq_umi
    for first, n in ((0, 2000), (123456789, 500)):
        want = make_fastq_umi(n=n, length=37, seed=9, first=first)
        got = ctx.synth("umi", n, 37, 9, first=first).download().tobytes()
        assert got == want
        # the DNA and quality lines are those of kind 0
        plain = synth.make_fastq(kind="illumina", n=n, length=37, seed=9, first=first).split(b"\n")
        assert [l for i, l in enumerate(got.split(b"\n")) if i % 4] == [l for i, l in enumerate(plain) if i % 4]


CASES = {
    "umi": lambda: umi_fastq(12000, length=20),
    "lengths_0_1_255": lambda: fastq_of(varlen_names()),
    "first": lambda: fastq_of(position_names("first")),
    "middle": lambda: fastq_of(position_names("middle")),
    "last": lambda: fastq_of(position_names("last")),
    "two_strings": lambda: fastq_of(two_string_names()),
    "width1": lambda: fastq_of(width_names(1)),
    "width2": lambda: fastq_of(width_names(2)),
    "width4": lambda: fastq_of(width_names(4)),
    "width8": lambda: fastq_of(width_names(8)),
    "late": lambda: fastq_of(late_names(), length=6),
    "long_names": lambda: fastq_of(long_names()),
}
_cache = {}


def _case(name):
    if name not in _cache:
        _cache[name] = CASES[name]()
    return _cache[name]


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_encode_and_decode_match_the_oracle(ctx, name):
    from oracle import uq_strings as lit
    from uq_b200 import host
    fq = _case(name)
    for mix in MIXES:
        ctxt = "%s %r" % (name, mix)
        want, want_cfg = lit.encode(fq, **mix)
        assert any(c["format"] == "strings" for c in want_cfg["QNAME_columns"]), ctxt
        got, cfg = host.encode(fq, ctx=ctx, **mix)
        assert_members_equal(got, want, ctxt)
        assert_config_equal(cfg, want_cfg, ctxt)
        text = host.decode(got, cfg, ctx=ctx).tobytes()
        stages = {}
        fqd = ctx.load_fastq(fq)
        dm, _ = host.encode_device(ctx, fqd, stages=stages, **mix)
        dt = host.decode_members_device(ctx, dm, cfg)
        dtext = dt.download().tobytes()
        dm.free(); dt.free(); fqd.free()
        for a in [stages["dna"], stages["qual"]] + stages["cols"]:
            a.free()
        assert dtext == text, ctxt
        if mix["sort"] == "None":
            assert text == fq, ctxt
        else:
            assert records_multiset(text) == records_multiset(fq), ctxt
            assert text == lit.decode(want, want_cfg), ctxt


def _np_rows(cols, kinds):
    parts = []
    for c, k in zip(cols, kinds):
        b = c.view(np.uint8).reshape(len(c), -1)
        parts.append(b if k else b[:, ::-1])
    return np.ascontiguousarray(np.concatenate(parts, axis=1))


@pytest.mark.gpu
@pytest.mark.parametrize("widths", [(4, 3, 1, 2), (1, 8, 5, 2, 8), (2, 60, 4), (8, 100, 1), (4, 255)])
def test_columns_rows_ex_against_numpy(ctx, widths):
    """kind 1 = bytes as they are, kind 0 = integer (big-endian in the row): staged (rows <= 64 B) and generic path"""
    rng = np.random.default_rng(sum(widths))
    n = 70001
    cols, kinds = [], []
    for i, w in enumerate(widths):
        if w in (1, 2, 8) and i % 2 == 0 or w == 4 and i == 0:
            cols.append(rng.integers(0, 2 ** (8 * w) - 1, size=n, dtype=np.uint64).astype("u%d" % w))
            kinds.append(0)
        else:
            cols.append(rng.integers(0, 256, size=(n, w), dtype=np.uint8).reshape(-1).view("S%d" % w))
            kinds.append(1)
    dcols = [ctx.upload(c.view(np.uint8).reshape(n, -1)) for c in cols]
    rows = ctx.columns_to_rows(dcols, kinds)
    want = _np_rows(cols, kinds)
    assert rows.width == sum(widths)
    assert np.array_equal(rows.download().reshape(n, -1), want)
    back = ctx.rows_to_columns(rows, list(widths), kinds)
    for c, b in zip(cols, back):
        assert np.array_equal(b.download().reshape(-1), c.view(np.uint8).reshape(-1))
    for a in dcols + back + [rows]:
        a.free()


@pytest.mark.gpu
@pytest.mark.parametrize("widths", [(1, 2, 4), (8, 8, 8, 8, 8, 8, 8, 8, 8), (2, 2)])
def test_columns_rows_ex_all_integer_equals_old_entry_points(ctx, widths):
    rng = np.random.default_rng(3)
    n = 50000
    cols = [ctx.upload(rng.integers(0, 2 ** (8 * w) - 1, size=n, dtype=np.uint64).astype("u%d" % w)) for w in widths]
    old = ctx.columns_to_rows(cols)
    new = ctx.columns_to_rows(cols, [0] * len(cols))
    assert old.first_difference(new) == -1
    b_old = ctx.rows_to_columns(old, list(widths))
    b_new = ctx.rows_to_columns(old, list(widths), [0] * len(cols))
    for a, b, c in zip(b_old, b_new, cols):
        assert a.first_difference(b) == -1 and a.first_difference(c) == -1
    for a in cols + b_old + b_new + [old, new]:
        a.free()


@pytest.mark.gpu
def test_mixfeed_serves_every_mix_like_a_fresh_encode(ctx):
    from uq_b200 import host
    fq = umi_fastq(11000, length=24, seed=12)
    feed = host.MixFeed(ctx, ctx.load_fastq(fq))
    try:
        for sort in ("None", "DNA", "QUAL", "QNAME"):
            for raw in (None, ["QNAME"], ["DNA", "QUAL"], ["DNA", "QUAL", "QNAME"]):
                for pattern in (None, ["2.2", "1.1"]):
                    want, want_cfg = host.encode(fq, ctx=ctx, sort=sort, raw=raw, pattern=pattern)
                    got = feed.members(sort, raw, pattern)
                    assert_members_equal(got, want, "feed %s %r %r" % (sort, raw, pattern))
                    assert_config_equal(feed.config(sort, raw, pattern), want_cfg)
    finally:
        feed.free()


def _sharded(world, fq, kw):
    from uq_b200 import multigpu as mg
    recs = [b"\n".join(r) + b"\n" for r in _records(fq)]
    n = len(recs)
    cuts = [0] + [n * (k + 1) // world for k in range(world - 1)] + [n]
    cuts[1] = max(cuts[1], min(n, 10001))
    for k in range(2, world):
        cuts[k] = max(cuts[k], cuts[k - 1] + 1)

    def body(c, comm):
        fqd = c.load_fastq(b"".join(recs[cuts[comm.rank]:cuts[comm.rank + 1]]))
        res, cfg = mg.encode_sharded(c, comm, fqd, **kw)
        members = mg.assemble(comm, res)
        res.free(); fqd.free()
        return members, cfg
    out = mg.run_local(world, body)
    assert len({json.dumps(c, sort_keys=True, default=str) for _, c in out}) == 1
    return out[0]


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_encode_equals_single_gpu(ctx, world):
    """includes a file whose longest string token lies on the last rank (every rank must pad to the global W)"""
    from uq_b200 import host, multigpu as mg
    rng = random.Random(11)
    names = ["s:%d:%s" % (i, _word(rng, rng.randrange(3, 10))) for i in range(24000)]
    names[23990] = "s:23990:" + _word(rng, 90)
    files = [umi_fastq(24000, length=20, seed=13), fastq_of(names)]
    for fq in files:
        for kw in (dict(sort="QNAME"), dict(sort="DNA", raw=["QNAME"]), dict(sort="None", raw=["QNAME"])):
            want, want_cfg = host.encode(fq, ctx=ctx, **kw)
            got, cfg = _sharded(world, fq, kw)
            assert_members_equal(got, want, "world %d %r" % (world, kw))
            assert json.loads(json.dumps(cfg)) == json.loads(json.dumps(want_cfg))
            parts = mg.run_local(world, lambda c, comm: bytes(mg.decode_sharded(c, comm, want, want_cfg)[0]))
            text = b"".join(parts)
            assert text == host.decode(want, want_cfg, ctx=ctx).tobytes()
            if kw["sort"] == "None":
                assert text == fq


@pytest.mark.gpu
def test_cli_encode_decode_and_peek(tmp_path):
    fq = umi_fastq(15000, length=30, seed=14)
    src = tmp_path / "umi.fastq"
    src.write_bytes(fq)
    env = dict(os.environ, PYTHONPATH=ROOT)
    out = tmp_path / "umi.uQ"
    r = subprocess.run([sys.executable, "-m", "uq_b200.uq", "-i", str(src), "-o", str(out)], env=env, cwd=ROOT,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 0 and out.is_file(), r.stdout.decode() + r.stderr.decode()
    d = subprocess.run([sys.executable, "-m", "uq_b200.uq", "-i", str(out), "--decode"], env=env, cwd=ROOT,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert d.returncode == 0, d.stderr.decode()
    assert d.stdout == fq
    p = subprocess.run([sys.executable, "-m", "uq_b200.uq", "-i", str(src), "--peek"], env=env, cwd=ROOT,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert p.returncode == 0, p.stderr.decode()
    assert '"format": "strings"' in p.stdout.decode()


def _device_members_equal(a, b):
    assert sorted(a.items) == sorted(b.items)
    for k in a.items:
        x, y = a.items[k][0], b.items[k][0]
        assert (x.n, x.width) == (y.n, y.width), k
        assert x.first_difference(y) == -1, k


@pytest.mark.gpu
def test_full_size_umi_resident_in_hbm(ctx):
    """100 M kind-4 reads: encode -> decode -> encode gives the same members; the unsorted raw decode is the input; the
    unique QNAME rows are strictly ascending in the E1 order"""
    from uq_b200 import host
    n = 100_000_000
    src = ctx.synth("umi", n, 150, 20260)
    fq = ctx.adopt_fastq(src)
    try:
        dm, cfg = host.encode_device(ctx, fq, sort="None", raw=["DNA", "QUAL", "QNAME"])
        assert cfg["QNAME_columns"][-1]["format"] == "strings" and cfg["QNAME_columns"][-1]["dtype"] == "|S12"
        text = host.decode_members_device(ctx, dm, cfg)
        dm.free()
        assert text.nbytes == src.nbytes and text.first_difference(src) == -1
        text.free()
        for sort in ("QNAME", "DNA"):
            dm, cfg = host.encode_device(ctx, fq, sort=sort)
            text = host.decode_members_device(ctx, dm, cfg)
            fq2 = ctx.adopt_fastq(text)
            dm2, cfg2 = host.encode_device(ctx, fq2, sort=sort)
            _device_members_equal(dm, dm2)
            assert cfg2 == cfg
            dm2.free(); fq2.free(); text.free()
            cols = [dm.items[m["name"]][0].download(dtype=np.dtype(m["dtype"])).reshape(-1) for m in cfg["QNAME_columns"]]
            less = np.zeros(len(cols[0]) - 1, dtype=bool)
            eq = np.ones(len(cols[0]) - 1, dtype=bool)
            for c in cols:
                less |= eq & (c[:-1] < c[1:])
                eq &= c[:-1] == c[1:]
            assert less.all(), "unique QNAME rows not strictly ascending (%s)" % sort
            dm.free()
    finally:
        fq.free()
        src.free()
