"""--verify: the encode decoded on the device and compared with its input record by record (host.verify_device,
k_verify_records, the permutation check).  Every device report is checked against np_verify, a numpy record splitter and
per-field comparison, on the same input, decoded text and order."""
import ctypes
import io
import os
import subprocess
import sys
import tarfile

import numpy as np
import pytest

from conftest import ROOT, golden_case, load_manifest

FIELDS = 4
CASES = sorted(load_manifest())


# ------------------------------------------------------------------------------------------------
# numpy reference
# ------------------------------------------------------------------------------------------------
def _records(buf):
    """bytes -> (uint8 array, int64 [n][5] line starts of every record; column 4 = start of the next record)"""
    a = np.frombuffer(buf, dtype=np.uint8)
    nl = np.flatnonzero(a == 10)
    assert len(nl) % 4 == 0
    off = np.concatenate(([0], nl + 1)).astype(np.int64)
    n = len(nl) // 4
    return a, off[np.arange(n)[:, None] * 4 + np.arange(5)]


def np_missing(order, n):
    """smallest value in [0, n) that order does not hold, -1 if none"""
    o = np.asarray(order, dtype=np.int64)
    seen = np.zeros(n, dtype=bool)
    seen[o[(o >= 0) & (o < n)]] = True
    miss = np.flatnonzero(~seen)
    return int(miss[0]) if len(miss) else -1


def np_verify(src, text, order=None, chunk_bytes=1 << 25):
    """decoded record i of `text` against input record order[i] of `src` (identity without an order): per field
    (0 name, 1 sequence, 2 '+' line, 3 quality) the rows whose line differs, the first such row and its input record.
    An order value outside the input is a difference in every field."""
    sa, so = _records(src)
    ta, to = _records(text)
    n, k = len(so), len(to)
    o = np.arange(k, dtype=np.int64) if order is None else np.asarray(order, dtype=np.int64)[:k]
    valid = o < n
    oi = np.where(valid, o, 0)
    S, T = so[oi], to
    lenbad = np.diff(S, axis=1) != np.diff(T, axis=1)
    bad = np.zeros((k, FIELDS), dtype=bool)
    bad[~valid] = True
    bad |= lenbad & valid[:, None]
    whole = np.flatnonzero(valid & ~lenbad.any(axis=1))
    if not (order is None and len(sa) == len(ta) and np.array_equal(sa, ta)):      # equal texts: equal records
        rl = S[whole, 4] - S[whole, 0]
        i = 0
        while i < len(whole):
            j = i + max(1, int(np.searchsorted(np.cumsum(rl[i:]), chunk_bytes)))
            rows, lens = whole[i:j], rl[i:j]
            ob = np.concatenate(([0], np.cumsum(lens)))
            pos = np.arange(ob[-1], dtype=np.int64)
            rep = np.repeat(np.arange(len(rows)), lens)
            d = np.flatnonzero(sa[S[rows, 0][rep] + pos - ob[rep]] != ta[T[rows, 0][rep] + pos - ob[rep]])
            if len(d):
                rr = rep[d]
                rel = d - ob[rr]
                b = S[rows[rr]] - S[rows[rr], :1]
                field = (rel >= b[:, 1]).astype(int) + (rel >= b[:, 2]) + (rel >= b[:, 3])
                bad[rows[rr], field] = True
            i = j
    for r in np.flatnonzero(valid & lenbad.any(axis=1)):                          # lines compared one by one
        for f in range(FIELDS):
            if not lenbad[r, f]:
                bad[r, f] |= not np.array_equal(sa[S[r, f]:S[r, f + 1]], ta[T[r, f]:T[r, f + 1]])
    first = [int(np.argmax(bad[:, f])) if bad[:, f].any() else -1 for f in range(FIELDS)]
    return dict(records=k, differ=[int(x) for x in bad.sum(axis=0)], first_row=first,
                first_src=[int(o[r]) if r >= 0 else -1 for r in first])


def _core(report):
    return {k: report[k] for k in ("records", "differ", "first_row", "first_src")}


def fastq_of(recs):
    return b"".join(b"%s\n%s\n%s\n%s\n" % tuple(r) for r in recs)


def simple_records(n, length=50, seed=3, names=None):
    """records without N (no N-trick: a changed DNA code always changes the decoded base)"""
    rng = np.random.default_rng(seed)
    dna = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=(n, length))]
    qual = rng.integers(53, 74, size=(n, length)).astype(np.uint8)
    names = names or [b"@SIM:1:FC:%d:%d" % (1 + i % 3, 1000 + i) for i in range(n)]
    return [(names[i], dna[i].tobytes(), b"+", qual[i].tobytes()) for i in range(n)]


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def test_np_verify_each_field_alone_and_together():
    recs = simple_records(6)
    src = fastq_of(recs)
    clean = np_verify(src, src)
    assert clean == dict(records=6, differ=[0, 0, 0, 0], first_row=[-1] * 4, first_src=[-1] * 4)
    for f, change in enumerate([lambda r: r[:-1] + b"9", lambda r: b"C" + r[1:], lambda r: r + b"name", lambda r: r[:-1]]):
        bad = [list(r) for r in recs]
        bad[4][f] = change(bad[4][f])
        rep = np_verify(src, fastq_of(bad))
        want = [0] * 4
        want[f] = 1
        assert rep["differ"] == want and rep["first_row"][f] == 4 and rep["first_src"][f] == 4, (f, rep)
    bad = [list(r) for r in recs]
    bad[2][0] = b"@x"                       # name shorter, sequence changed: both fields, bytes compared line by line
    bad[2][1] = b"G" + bad[2][1][1:] if bad[2][1][:1] != b"G" else b"A" + bad[2][1][1:]
    bad[5][3] = bad[5][3][:-1] + b"!"
    rep = np_verify(src, fastq_of(bad))
    assert rep["differ"] == [1, 1, 0, 1] and rep["first_row"] == [2, 2, -1, 5] and rep["first_src"] == [2, 2, -1, 5]


def test_np_verify_under_an_order():
    recs = simple_records(7, seed=9)
    src = fastq_of(recs)
    order = np.array([3, 0, 6, 1, 5, 2, 4])
    text = fastq_of([recs[i] for i in order])
    assert np_verify(src, text, order)["differ"] == [0, 0, 0, 0]
    assert np_verify(src, text, np.arange(7))["differ"][1] > 0           # the identity does not fit a shuffled text
    assert np_verify(src, text)["differ"] == np_verify(src, text, np.arange(7))["differ"]
    swapped = order.copy()
    swapped[[1, 5]] = swapped[[5, 1]]
    rep = np_verify(src, text, swapped)
    assert rep["first_row"][1] == 1 and rep["first_src"][1] == 2 and rep["differ"][1] == 2
    rep = np_verify(src, text, np.array([3, 0, 6, 1, 5, 2, 99]))
    assert rep["differ"] == [1, 1, 1, 1] and rep["first_src"] == [99] * 4
    assert np_missing(order, 7) == -1 and np_missing([3, 0, 6, 1, 5, 3, 4], 7) == 2


def test_cli_parser_accepts_verify_and_refuses_it_with_decode_or_peek(tmp_path, capsys):
    from uq_b200 import uq
    a = uq.build_parser().parse_args(["-i", "x.fastq", "--sort", "DNA", "--verify"])
    assert a.verify and not uq.build_parser().parse_args(["-i", "x.fastq"]).verify
    src = tmp_path / "in.fastq"
    src.write_bytes(fastq_of(simple_records(4)))
    for extra in ("--decode", "--peek"):
        assert uq.main(["-i", str(src), "--verify", extra]) == 0          # an option error: printed, no device touched
        out = capsys.readouterr().out
        assert "--verify" in out and extra in out
    assert not (tmp_path / "in.fastq.uQ").exists()


def test_verify_report_size_matches_the_header(tmp_path):
    from uq_b200 import _lib
    src = tmp_path / "size.c"
    src.write_text('#include <stdio.h>\n#include "uqb200.h"\nint main(void){printf("%zu\\n",sizeof(uqb_verify_report));return 0;}\n')
    exe = tmp_path / "size"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = int(subprocess.run([str(exe)], stdout=subprocess.PIPE, text=True, check=True).stdout)
    assert got == ctypes.sizeof(_lib.VerifyReport) == 8 + 3 * 32


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    from uq_b200.device import Context
    c = Context(0)
    yield c
    c.close()


class Run:
    """one encode on the device, verified; keeps what the reference comparison needs"""

    def __init__(self, ctx, fastq, batch_rows=1 << 24, tamper=None, **kw):
        from uq_b200 import host
        self.ctx = ctx
        self.fq = ctx.load_fastq(fastq) if not hasattr(fastq, "device_ptr") else ctx.adopt_fastq(fastq)
        self.members, self.config = host.encode_device(ctx, self.fq, **kw)
        if tamper is not None:
            tamper(self)
        self.report = host.verify_device(ctx, self.fq, self.members, self.config, batch_rows=batch_rows)
        self.order = None if self.members.order is None else self.members.order.download(dtype=np.uint32)

    def text(self):
        from uq_b200 import host
        t = host.decode_members_device(self.ctx, self.members, self.config)
        out = t.download().tobytes()
        t.free()
        return out

    def check(self, src):
        """the device report equals np_verify on the input, the decoded text and the order"""
        want = np_verify(src, self.text(), self.order)
        assert _core(self.report) == want, (self.report, want)
        assert self.report["missing"] == (-1 if self.order is None else np_missing(self.order, len(self.order)))
        return want

    def free(self):
        self.members.free()
        self.fq.free()


def _clean(rep, n):
    assert rep["records"] == n and rep["differ"] == [0, 0, 0, 0] and rep["missing"] == -1, rep
    assert rep["first_row"] == [-1] * 4 and rep["lines"] == {}


def _kernels(ctx):
    return set(ctx.timing_report())


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_golden_cases_verify_clean(ctx, name):
    fq, _, kw = golden_case(name)
    r = Run(ctx, fq, **kw)
    n = r.config["reads"]
    _clean(r.report, n)
    r.check(fq)
    if kw["sort"] not in (None, "None"):
        assert r.order is not None and not np.array_equal(r.order, np.arange(n))
    else:
        assert r.order is None
    r.free()


MIXES = {"raw": ["DNA", "QUAL", "QNAME"], "keyed": None, "mixed": ["QUAL"]}
PATTERNS = [("0.1", "0.1"), ("2.2", "1.2"), ("3.1", "0.2")]


@pytest.fixture(scope="module")
def synth2m(ctx):
    n = 2_000_000
    dev = ctx.synth("genome", n, 150, 2026, genome=200_000, pool=400_000)
    yield n, dev, dev.download().tobytes(), {}
    dev.free()


@pytest.mark.gpu
@pytest.mark.parametrize("sort", ["None", "DNA", "QUAL", "QNAME"])
def test_two_million_reads_every_mix_verifies_clean(ctx, synth2m, sort):
    """2 M reads: --sort None / DNA / QUAL / QNAME x all raw / all keyed / mixed x three pattern pairs.  For one sort
    every mix decodes to the same text under the same order, so one np_verify per sort covers all nine reports: each
    case's decoded text is compared with the first case's on the device and its order with the first case's order."""
    n, dev, src, _ = synth2m
    first_text, first_order, want = None, None, None
    for mix, raw in MIXES.items():
        for pattern in PATTERNS:
            ctx.timing(True)
            ctx.timing_reset()
            r = Run(ctx, dev, sort=sort, raw=raw, pattern=list(pattern))
            k = _kernels(ctx)
            ctx.timing(False)
            _clean(r.report, n)
            assert "k_verify_records" in k
            assert ("k_perm_mark" in k and "k_perm_missing" in k) == (sort != "None"), k
            from uq_b200 import host
            text = host.decode_members_device(ctx, r.members, r.config)
            if first_text is None:
                first_text, first_order = text, r.order
                want = np_verify(src, text.download().tobytes(), r.order)
            else:
                assert text.first_difference(first_text) == -1, (mix, pattern)
                assert (r.order is None) == (first_order is None)
                assert r.order is None or np.array_equal(r.order, first_order)
                text.free()
            assert _core(r.report) == want, (mix, pattern)
            r.free()
    first_text.free()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,sort", [("ont", "QUAL"), ("ont", "None"), ("umi", "QNAME"), ("renamed", "DNA"), ("mixed", "None"),
                                       ("mixed", "QNAME")])
def test_variable_length_and_qname_kinds_verify_clean(ctx, kind, sort):
    """kind 3 (variable length), kind 4 ('strings' QNAME column, E1), kinds 5 / 6 (one QNAME column, E2)"""
    from oracle import synth
    if kind == "ont":
        dev = ctx.synth("ont", 3000, (50, 4000), 31, len_table=synth.ont_length_table(50, 4000))
    else:
        dev = ctx.synth(kind, 200_000, 100, 32)
    src = dev.download().tobytes()
    r = Run(ctx, dev, sort=sort)
    if kind == "umi":
        assert any(c["format"] == "strings" for c in r.config["QNAME_columns"])
    if kind in ("renamed", "mixed"):
        assert r.config["QNAME_separators"] == "" and len(r.config["QNAME_columns"]) == 1
    _clean(r.report, r.config["reads"])
    r.check(src)
    r.free()
    dev.free()


def plus_name_records(n=3000, at=(5, 997, 1800), seed=7):
    recs = simple_records(n, seed=seed)
    for i in at:
        recs[i] = (recs[i][0], recs[i][1], b"+" + recs[i][0][1:], recs[i][3])
    return recs


def zero_padded_records(n=3000, start=1234, seed=8):
    """names '@r:<a>:<b>' whose middle column is written with leading zeros from record `start` on"""
    names = [b"@r:%d:%d" % (i % 700, i % 5) if i < start else b"@r:%04d:%d" % (i % 700, i % 5) for i in range(n)]
    return simple_records(n, seed=seed, names=names)


@pytest.mark.gpu
@pytest.mark.parametrize("sort", ["None", "DNA"])
def test_lossy_plus_lines_are_reported(ctx, sort):
    at = (5, 997, 1800)
    src = fastq_of(plus_name_records(at=at))
    r = Run(ctx, src, sort=sort)
    want = r.check(src)
    rep = r.report
    assert rep["differ"] == [0, 0, 3, 0] and want["differ"] == [0, 0, 3, 0]
    rows = [int(np.flatnonzero(r.order == i)[0]) for i in at] if r.order is not None else list(at)
    assert rep["first_row"][2] == min(rows) and rep["first_src"][2] == at[int(np.argmin(rows))]
    inp, dec = rep["lines"][2]
    assert dec == b"+" and inp == b"+" + src.split(b"\n")[4 * rep["first_src"][2]][1:]
    r.free()


@pytest.mark.gpu
@pytest.mark.parametrize("sort", ["None", "DNA"])
def test_lossy_zero_padded_integer_column_is_reported(ctx, sort):
    start = 1234
    src = fastq_of(zero_padded_records(start=start))
    r = Run(ctx, src, sort=sort)
    assert r.config["QNAME_columns"][1]["format"] == "integers"
    want = r.check(src)
    rep = r.report
    assert rep["differ"] == [3000 - start, 0, 0, 0] == want["differ"]
    if r.order is None:
        assert rep["first_row"][0] == start and rep["first_src"][0] == start
    inp, dec = rep["lines"][0]
    s = rep["first_src"][0]
    assert inp == b"@r:%04d:%d" % (s % 700, s % 5) and dec == b"@r:%d:%d" % (s % 700, s % 5)
    r.free()


def _set_bytes(ctx, arr, offset, data):
    tmp = ctx.upload(np.frombuffer(data, dtype=np.uint8))
    ctx.copy_in(arr, offset, tmp.device_ptr.value, len(data))
    ctx.sync()
    tmp.free()


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", ["0.1", "0.2"])
def test_tampered_raw_dna_byte_is_reported(ctx, pattern):
    src = fastq_of(simple_records(4000, seed=11))
    row = 2345

    def flip(run):
        stream, _, (n, width, p) = run.members.items["DNA.raw"]
        pos = row * width if p == "0.1" else row                # byte 0 of the row: row-major, or column 0 of the transpose
        b = stream.download().reshape(-1)[pos]
        _set_bytes(ctx, stream, pos, bytes([b ^ 0x03]))
    r = Run(ctx, src, sort="None", raw=["DNA", "QUAL", "QNAME"], pattern=[pattern, "0.1"], tamper=flip)
    r.check(src)
    assert r.report["differ"] == [0, 1, 0, 0] and r.report["first_row"][1] == row and r.report["first_src"][1] == row
    r.free()


@pytest.mark.gpu
def test_tampered_keyed_qual_row_reports_every_row_that_points_to_it(ctx):
    recs = simple_records(5000, length=20, seed=12)
    recs = [(a, b, c, recs[i % 40][3]) for i, (a, b, c, _) in enumerate(recs)]        # 40 distinct quality lines
    src = fastq_of(recs)
    state = {}

    def swap_row(run):
        stream, _, (n, width, p) = run.members.items["QUAL"]
        key = run.members.items["QUAL.key"][0].download(dtype=np.dtype(run.members.items["QUAL.key"][2])).astype(np.int64)
        u = int(key[17])
        other = (u + 1) % n
        uniq = stream.download().reshape(n, width)
        _set_bytes(ctx, stream, u * width, uniq[other].tobytes())
        state["count"], state["first"] = int((key == u).sum()), int(np.argmax(key == u))
    r = Run(ctx, src, sort="DNA", tamper=swap_row)
    r.check(src)
    rep = r.report
    assert rep["differ"] == [0, 0, 0, state["count"]] and rep["first_row"][3] == state["first"]
    r.free()


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["swap", "repeat"])
def test_tampered_order_is_reported(ctx, how):
    src = fastq_of(simple_records(3000, seed=13))
    state = {}

    def change(run):
        o = run.members.order.download(dtype=np.uint32).copy()
        state["old"] = o.copy()
        if how == "swap":
            o[[10, 2500]] = o[[2500, 10]]
        else:
            o[2500] = o[10]
        _set_bytes(ctx, run.members.order, 0, o.tobytes())
    r = Run(ctx, src, sort="DNA", tamper=change)
    want = r.check(src)
    old = state["old"]
    if how == "swap":
        assert r.report["missing"] == -1
        assert r.report["first_row"][1] == 10 and r.report["first_src"][1] == int(old[2500]) and want["differ"][1] == 2
    else:
        assert r.report["missing"] == int(old[2500])
        assert r.report["first_row"][1] == 2500 and r.report["first_src"][1] == int(old[10]) and want["differ"][1] == 1
    r.free()


@pytest.mark.gpu
@pytest.mark.parametrize("sort,raw,pattern", [("None", ["DNA", "QNAME"], ["0.1", "0.1"]), ("DNA", None, ["2.2", "1.2"]),
                                              ("QNAME", ["DNA", "QUAL"], ["3.1", "0.2"])])
def test_batch_size_does_not_change_the_report(ctx, sort, raw, pattern):
    """mismatches on both sides of the 997-row batch boundaries: identical reports at 1, 997, 2^20 and n rows"""
    recs = plus_name_records(n=2500, at=(3, 996, 997, 1993, 1994, 2400))
    recs = [(b"@SIM:1:FC:%d:%05d" % (1 + i % 3, 1000 + i) if 990 <= i < 1000 else a, b, c, d) for i, (a, b, c, d) in enumerate(recs)]
    src = fastq_of(recs)
    reports = []
    for batch in (1, 997, 1 << 20, 2500):
        r = Run(ctx, src, batch_rows=batch, sort=sort, raw=raw, pattern=pattern)
        if batch == 997:
            r.check(src)
        reports.append(r.report)
        r.free()
    assert reports[0]["differ"][2] == 6 and reports[0]["differ"][0] > 0
    assert all(x == reports[0] for x in reports[1:])


@pytest.mark.gpu
def test_config1_full_size_sort_dna_keyed_verifies_clean(ctx):
    """configs[1] at full size: 100 M reads x 150 bp, --sort DNA, keyed tables, verified batch by batch"""
    from uq_b200 import host
    n = 100_000_000
    used, free, total = ctx.mem_info()
    if total - used < 150 << 30:
        pytest.skip("needs ~150 GB of free HBM")
    dev = ctx.synth("genome", n, 150, 1002, genome=10_000_000, pool=n // 5)
    fq = ctx.adopt_fastq(dev)
    m, cfg = host.encode_device(ctx, fq, sort="DNA")
    batch = host.verify_batch_rows(ctx, fq, m, cfg)
    assert batch >= 1 << 20
    ctx.timing(True)
    ctx.timing_reset()
    rep = host.verify_device(ctx, fq, m, cfg, batch_rows=batch)
    k = ctx.timing_report()
    ctx.timing(False)
    _clean(rep, n)
    assert k["k_verify_records"][0] == -(-n // batch) and k["k_perm_mark"][0] == 1
    m.free(); fq.free(); dev.free()


def _members_of(data):
    tar = tarfile.open(fileobj=io.BytesIO(data))
    return {x: tar.extractfile(x).read() for x in tar.getnames()}


def _cli(args):
    env = dict(os.environ, PYTHONPATH=ROOT)
    return subprocess.run([sys.executable, "-m", "uq_b200.uq"] + args, env=env, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c2_keyed_sortDNA", "c1_raw_p12_01"])
def test_cli_verify_writes_the_reference_members(tmp_path, name):
    fq, uq, _ = golden_case(name)
    src, out = tmp_path / "in.fastq", tmp_path / "out.uQ"
    src.write_bytes(fq)
    r = _cli(["-i", str(src), "-o", str(out), "--verify"] + load_manifest()[name]["options"])
    text = r.stdout.decode()
    assert r.returncode == 0 and out.is_file(), text + r.stderr.decode()
    assert "Verified: all %d records" % (fq.count(b"\n") // 4) in text
    got, want = _members_of(out.read_bytes()), _members_of(uq)
    assert sorted(got) == sorted(want)
    for k in want:
        if k != "config.json":
            assert got[k] == want[k], k


@pytest.mark.gpu
def test_cli_verify_refuses_a_lossy_file(tmp_path):
    recs = plus_name_records(n=2000, at=(1500,))
    src, out = tmp_path / "in.fastq", tmp_path / "out.uQ"
    src.write_bytes(fastq_of(recs))
    r = _cli(["-i", str(src), "-o", str(out), "--verify", "--sort", "DNA"])
    text = r.stdout.decode()
    assert r.returncode == 1, text + r.stderr.decode()
    assert not out.exists()
    assert "+ line: 1 records differ" in text and "input record 1500" in text
    assert repr(b"+" + recs[1500][0][1:]) in text and "decoded: b'+'" in text and "Q13" in text


@pytest.mark.gpu
def test_encode_without_verify_launches_no_verify_kernel(ctx):
    from uq_b200 import host
    fq, _, kw = golden_case("c2_keyed_sortDNA")
    ctx.timing(True)
    ctx.timing_reset()
    members, cfg = host.encode(fq, ctx=ctx, **kw)
    k = _kernels(ctx)
    ctx.timing(False)
    assert not k & {"k_verify_records", "k_perm_mark", "k_perm_missing"}, k
