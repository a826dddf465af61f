"""QNAMEs that do not split into columns (declared extension E2, DESIGN section 4): where the reference's layout step
refuses a file (Q6, Q8, Q11, separators in another order) or a record does not hold the separators in their order,
the names are stored as ONE column between the longest common prefix and suffix.  The host decision and the oracle
run without a GPU; the device encode and decode, the --test feed, the sharded path, the CLI and 100 M-read inputs are
checked on the GPU against the oracle (oracle/uq_names.py)."""
import json
import os
import random
import subprocess
import sys

import pytest

from conftest import ROOT, assert_config_equal, assert_members_equal, records_multiset
from emu import emu_colstats, emu_stats
from test_host_logic import _fastq, _rand_names

MIXES = [dict(sort=s, raw=r) for s in ("None", "DNA", "QNAME") for r in (None, ["QNAME"])]


# ------------------------------------------------------------------------------------------------
# inputs: one per refusal kind and the layout / typing corner cases
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


def _word(rng, n, alphabet="ACGT"):
    return "".join(rng.choice(alphabet) for _ in range(n))


def q6_names(n=400):
    """renamed reads: no character with a constant count"""
    return ["SRR1234.%d" % (i + 1) for i in range(n)]


def order_names(n=300, seed=1):
    """':' and '_' occur once in every name, the last name has them the other way round (uq.py:438-444)"""
    rng = random.Random(seed)
    out = ["x%d:%d_%d" % (i, rng.randrange(50), rng.randrange(9)) for i in range(n)]
    out[-1] = "x%d_%d:%d" % (n - 1, rng.randrange(50), rng.randrange(9))
    return out


def bad_record_names(n=300, seed=2, at=150):
    """first and last name agree, record `at` has the separators the other way round: the tokeniser flags it"""
    names = order_names(n, seed)
    names[-1] = "x%d:1_2" % (n - 1)
    names[at] = "x%d_3:4" % at
    return names


def q8_names(n=300):
    """a name that is a proper prefix of the running common prefix (the reference raises IndexError)"""
    names = ["read:1:%d" % i for i in range(n)]
    names[120] = "read:1"
    return names


def q11_names(n=300):
    """separators ':', '-', '_': the unescaped class ':-_' is a range that takes in the capitals"""
    return ["x%d:%d-%d_%d" % (i, i, i + 1, i + 2) for i in range(1, n + 1)]


def identical_names(n=200):
    return ["same:name 1"] * n


def prefix_equal_names(n=300):
    """one name is the common prefix itself: its middle is empty"""
    names = ["ab%d" % i for i in range(n)]
    names[77] = "ab"
    return names


def overlap_names(n=300, seed=3):
    """the common suffix 'zxy' of the names reaches into the common prefix '@xyz' of the first one ('@xyzxy' /
    '@xyz..zxy'): the suffix is clamped to the shortest remainder 'xy'"""
    rng = random.Random(seed)
    return ["xyzxy"] + ["xyz" + _word(rng, rng.randrange(6), "zq") + "zxy" for _ in range(n - 1)]


def canonical_int_names(n=400, seed=4):
    rng = random.Random(seed)
    return ["%d" % rng.randrange(-1000, 100000) for _ in range(n)]


def noncanonical_int_names(n=400, seed=5):
    """leading zeros: stored as text, never as integers (no Q9 loss)"""
    rng = random.Random(seed)
    return ["%05d" % rng.randrange(100000) for _ in range(n)]


def wide_names(width, n=200, seed=6):
    """middles of up to `width` bytes between '<' and '>'"""
    rng = random.Random(seed + width)
    out = ["<%s>" % _word(rng, rng.randrange(1, width + 1)) for _ in range(n)]
    out[17] = "<%s>" % _word(rng, width)
    return out


CASES = {
    "q6": lambda: fastq_of(q6_names()),
    "order": lambda: fastq_of(order_names()),
    "bad_record": lambda: fastq_of(bad_record_names()),
    "q8": lambda: fastq_of(q8_names()),
    "q11": lambda: fastq_of(q11_names()),
    "identical": lambda: fastq_of(identical_names()),
    "prefix_equal": lambda: fastq_of(prefix_equal_names()),
    "overlap": lambda: fastq_of(overlap_names()),
    "canonical_ints": lambda: fastq_of(canonical_int_names()),
    "noncanonical_ints": lambda: fastq_of(noncanonical_int_names()),
    "middle_255": lambda: fastq_of(wide_names(255)),
}
_cache = {}


def _case(name):
    if name not in _cache:
        _cache[name] = CASES[name]()
    return _cache[name]


def _records(fq):
    ls = fq.split(b"\n")[:-1]
    return [tuple(ls[i:i + 4]) for i in range(0, len(ls), 4)]


def emu_decision(fq):
    """host.decide_qname_columns on the CPU emulation of the device statistics -> (prefix, suffix, seps, columns,
    derive_qname_layout refused the file, a record did not split)"""
    from uq_b200 import host
    st, n = emu_stats(fq)
    seen = {}

    def scan(p, s, seps):
        cols, bad, dicts = emu_colstats(fq, len(p), len(s), seps)
        seen["dicts"] = dicts
        if seps:
            seen["bad"] = bad
        return cols, bad
    try:
        host.derive_qname_layout(st, n)
        refused = False
    except host.UQError:
        refused = True
    out = host.decide_qname_columns(st, n, scan, lambda plen: int(emu_colstats(fq, plen, 0, "")[0][0].min_len),
                                    lambda i: seen["dicts"][i])
    return out + (refused, seen.get("bad", -1) >= 0)


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("style", [0, 1, 2, 3])
def test_decision_equals_oracle_on_random_names(style):
    """the _rand_names sets of test_host_logic: every set the reference's layout step refuses gets an E2 layout whose
    prefix + middle + suffix rebuilds every name, and the whole decision equals oracle/uq_names.py"""
    from oracle import uq_literal as lit, uq_names, uq_strings
    rng = random.Random(1234 + style)
    e2 = 0
    for _ in range(400):
        names = _rand_names(rng, style)
        fq = _fastq(names)
        prefix, suffix, seps, columns, refused, bad = emu_decision(fq)
        lines, total = lit.split_lines(fq)
        want = uq_names.reference_layout(lines, total)
        if want is None:
            e2 += 1
            assert refused or bad, names
            assert seps == "" and [c["name"] for c in columns] == ["QNAME_1"], names
            assert (prefix, suffix) == uq_names.layout(lines, total), names
            toks = uq_names.tokens(lines, total, prefix, suffix)
            assert all(prefix + t + suffix == nm.decode("latin-1") for t, nm in zip(toks, names)), names
            assert columns == uq_names.pass2(toks), names
        else:
            assert not refused and not bad, names
            assert (prefix, suffix, seps) == want, names
            if seps:        # '' = none of the surviving separators occurs in the first and last name: not E2's ground
                assert columns == uq_strings.pass2(lines, total, prefix, suffix, seps), names
    assert e2 >= (5, 150, 1, 350)[style]


@pytest.mark.parametrize("name", sorted(CASES))
def test_inputs_take_e2_for_the_intended_reason(name):
    fq = _case(name)
    prefix, suffix, seps, columns, refused, bad = emu_decision(fq)
    assert seps == "" and len(columns) == 1
    assert bad if name == "bad_record" else refused
    want = {"q6": "integers", "canonical_ints": "integers", "noncanonical_ints": "strings", "middle_255": "strings",
            "identical": "mapping"}.get(name)
    if want:
        assert columns[0]["format"] == want, columns
    if name == "middle_255":
        assert columns[0]["dtype"] == "|S255"
    if name == "overlap":
        assert (prefix, suffix) == ("@xyz", "xy")
    if name == "prefix_equal":
        assert prefix == "@ab"


def test_wider_middle_is_refused():
    from oracle import uq_names
    from uq_b200 import host
    fq = fastq_of(wide_names(256))
    with pytest.raises(host.UQError, match="holds a token of 256 bytes"):
        emu_decision(fq)
    with pytest.raises(uq_names.UQError, match="holds a token of 256 bytes"):
        uq_names.encode(fq)


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_round_trip(name):
    from oracle import uq_names
    fq = _case(name)
    for mix in MIXES + [dict(sort="QUAL", raw=["DNA"])]:
        m, c = uq_names.encode(fq, **mix)
        assert c["QNAME_separators"] == "" and len(c["QNAME_columns"]) == 1
        text = uq_names.decode(m, c)
        if mix["sort"] == "None":
            assert text == fq, mix
        else:
            assert records_multiset(text) == records_multiset(fq), mix


def test_oracle_is_uq_strings_on_tokenisable_files():
    from oracle import uq_names, uq_strings
    from test_qname_strings import fastq_of as strings_fastq, two_string_names
    for fq in (strings_fastq(two_string_names()), fastq_of(["r:%d:%d" % (i % 7, i) for i in range(500)])):
        a, ca = uq_names.encode(fq, sort="QNAME")
        b, cb = uq_strings.encode(fq, sort="QNAME")
        assert_members_equal(a, b)
        assert_config_equal(ca, cb)


def test_synth_twins_take_e2():
    """the host generators of synth kinds 5 and 6 are E2 files: kind 5 an integers column, kind 6 strings"""
    from oracle import uq_names
    from oracle.synth_names import make_fastq_names
    for kind, fmt in (("renamed", "integers"), ("mixed", "strings")):
        fq = make_fastq_names(kind=kind, n=2500, length=20, seed=3)
        prefix, suffix, seps, columns, refused, bad = emu_decision(fq)
        assert refused and seps == "" and columns[0]["format"] == fmt, (kind, columns)
        m, c = uq_names.encode(fq)
        assert uq_names.decode(m, c) == fq


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
def test_device_synth_names_match_host(ctx):
    from oracle import synth
    from oracle.synth_names import make_fastq_names
    for kind in ("renamed", "mixed"):
        for first, n in ((0, 3000), (123456789, 700)):
            want = make_fastq_names(kind=kind, n=n, length=37, seed=9, first=first)
            got = ctx.synth(kind, n, 37, 9, first=first).download().tobytes()
            assert got == want, kind
            plain = synth.make_fastq(kind="illumina", n=n, length=37, seed=9, first=first).split(b"\n")
            assert [l for i, l in enumerate(got.split(b"\n")) if i % 4] == [l for i, l in enumerate(plain) if i % 4]


def _device_round_trip(ctx, fq, mix, cfg, text):
    from uq_b200 import host
    stages = {}
    fqd = ctx.load_fastq(fq)
    dm, _ = host.encode_device(ctx, fqd, stages=stages, **mix)
    dt = host.decode_members_device(ctx, dm, cfg)
    dtext = dt.download().tobytes()
    dm.free(); dt.free(); fqd.free()
    for a in [stages["dna"], stages["qual"]] + stages["cols"]:
        a.free()
    assert dtext == text


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_encode_and_decode_match_the_oracle(ctx, name):
    from oracle import uq_names
    from uq_b200 import host
    fq = _case(name)
    for mix in MIXES:
        ctxt = "%s %r" % (name, mix)
        want, want_cfg = uq_names.encode(fq, **mix)
        got, cfg = host.encode(fq, ctx=ctx, **mix)
        assert_members_equal(got, want, ctxt)
        assert_config_equal(cfg, want_cfg, ctxt)
        assert cfg["QNAME_separators"] == "" and len(cfg["QNAME_columns"]) == 1
        text = host.decode(got, cfg, ctx=ctx).tobytes()
        _device_round_trip(ctx, fq, mix, cfg, text)
        if mix["sort"] == "None":
            assert text == fq, ctxt
        else:
            assert records_multiset(text) == records_multiset(fq), ctxt
            assert text == uq_names.decode(want, want_cfg), ctxt


@pytest.mark.gpu
def test_wider_middle_is_refused_on_the_device(ctx):
    from uq_b200 import host
    with pytest.raises(host.UQError, match="holds a token of 256 bytes"):
        host.encode(fastq_of(wide_names(256)), ctx=ctx)


@pytest.mark.gpu
def test_mixfeed_serves_every_mix_like_a_fresh_encode(ctx):
    from oracle.synth_names import make_fastq_names
    from uq_b200 import host
    for fq in (make_fastq_names(kind="mixed", n=11000, length=24, seed=12), fastq_of(q8_names())):
        feed = host.MixFeed(ctx, ctx.load_fastq(fq))
        try:
            for sort in ("None", "DNA", "QUAL", "QNAME"):
                for raw in (None, ["QNAME"], ["DNA", "QUAL", "QNAME"]):
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
    """includes a record that does not split at the separators and lies on the last rank only: every rank switches"""
    from oracle.synth_names import make_fastq_names
    from uq_b200 import host, multigpu as mg
    late_bad = bad_record_names(n=24000, at=20000)
    files = [make_fastq_names(kind="renamed", n=24000, length=20, seed=13), fastq_of(late_bad),
             make_fastq_names(kind="mixed", n=24000, length=20, seed=14)]
    for fq in files:
        for kw in (dict(sort="QNAME"), dict(sort="DNA", raw=["QNAME"]), dict(sort="None", raw=["QNAME"])):
            want, want_cfg = host.encode(fq, ctx=ctx, **kw)
            assert want_cfg["QNAME_separators"] == ""
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
    fq = fastq_of(q8_names(n=3000))
    src = tmp_path / "q8.fastq"
    src.write_bytes(fq)
    env = dict(os.environ, PYTHONPATH=ROOT)
    out = tmp_path / "q8.uQ"
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
    assert '"QNAME_separators": ""' in p.stdout.decode()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,kw,fmt", [("renamed", dict(sort="QNAME"), "integers"),
                                         ("mixed", dict(sort="None", raw=["DNA", "QUAL", "QNAME"]), "strings")])
def test_full_size_names_resident_in_hbm(ctx, kind, kw, fmt):
    """100 M reads of kind 5 (keyed, sorted on the QNAME, which is the record order) and of kind 6 (raw, unsorted):
    the decode is the input, byte for byte, compared on the device"""
    from uq_b200 import host
    n = 100_000_000
    src = ctx.synth(kind, n, 150, 20260)
    fq = ctx.adopt_fastq(src)
    try:
        dm, cfg = host.encode_device(ctx, fq, **kw)
        col = cfg["QNAME_columns"]
        assert cfg["QNAME_separators"] == "" and len(col) == 1 and col[0]["format"] == fmt, col
        if kind == "renamed":
            assert cfg["QNAME_prefix"] == "@SRR0000001." and (col[0]["min"], col[0]["max"]) == (1, n)
            assert col[0]["dtype"] == "uint32"
        text = host.decode_members_device(ctx, dm, cfg)
        dm.free()
        assert text.nbytes == src.nbytes and text.first_difference(src) == -1
        text.free()
    finally:
        fq.free()
        src.free()
