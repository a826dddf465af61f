"""GPU parity tests: every stage of libuqb200.so through the C ABI against the oracle / the
reference-written golden containers.  Run on the B200 box with `pytest -m gpu`."""
import numpy as np
import pytest

from conftest import (assert_config_equal, assert_members_equal, golden_case, load_manifest,
                      records_multiset)
from emu import emu_colstats, emu_stats

pytestmark = pytest.mark.gpu

CASES = sorted(load_manifest())


@pytest.fixture(scope="module")
def ctx():
    from uq_b200.device import Context
    c = Context(0)
    yield c
    c.close()


def _line_offsets_ref(fq):
    a = np.frombuffer(fq, dtype=np.uint8)
    nl = np.flatnonzero(a == 10).astype(np.uint64) + 1
    return np.concatenate([np.zeros(1, np.uint64), nl])


def test_context_and_abi_version(ctx):
    """ABI 101: uqb_qname_scan, uqb_fastq_load_streamed, uqb_columns_to_rows and uqb_rows_to_columns take their
    optional arguments (col_mode; ref, ref_len, rbase; kinds) directly"""
    assert ctx.lib.uqb_version() == 101
    used, free, total = ctx.mem_info()
    assert total > 100 << 30, "expected a B200 with ~180 GB of HBM"


@pytest.mark.parametrize("case", ["c1_raw_p01_31", "c5_variable_raw", "c6_checkpoints"])
def test_split_matches_numpy(ctx, case):
    fq, _, _ = golden_case(case)
    for data in (fq, fq[:-1], fq + b"@tail-without-newline", fq[:len(fq) // 3]):
        d = ctx.load_fastq(data)
        info = d.split()
        ref = _line_offsets_ref(data)
        assert info.n_lines == len(ref) - 1
        assert info.status == (0 if (len(ref) - 1) % 4 == 0 else 1)
        got = d.line_offsets()
        assert np.array_equal(got, ref)
        d.free()


def test_split_empty_and_tiny(ctx):
    for data in (b"", b"\n", b"a", b"\n\n\n\n", b"@a\nA\n+\nI\n"):
        d = ctx.load_fastq(data)
        info = d.split()
        assert info.n_lines == data.count(b"\n")
        assert np.array_equal(d.line_offsets(), _line_offsets_ref(data))
        d.free()


@pytest.mark.parametrize("shape", ["even", "dense_tail", "no_newline", "odd_size"])
def test_split_single_pass_matches_numpy(ctx, shape):
    """files of 1 MB and more take the one-pass newline scan (k_newline_scan1): its look-back numbering, the capacity
    estimate from the head of the file, and the two-pass fallback when the tail is denser than the head"""
    rng = np.random.default_rng(11)
    if shape == "even":
        data = rng.integers(0, 64, size=9_000_001, dtype=np.uint8)            # a newline every 64 bytes on average
    elif shape == "dense_tail":
        # 70 MB: the first 66 MB (all 4096 sampled tiles) hold few newlines, the tail is dense -> the estimate overflows
        data = rng.integers(11, 255, size=70_000_000, dtype=np.uint8)
        data[::5000] = 10
        data[67_000_000:] = rng.integers(10, 12, size=3_000_000, dtype=np.uint8)      # 1.5 M newlines > the 1 M slack
    elif shape == "no_newline":
        data = rng.integers(11, 255, size=3_000_000, dtype=np.uint8)
    else:
        data = rng.integers(0, 32, size=4 * 16384 * 70 + 12345, dtype=np.uint8)
        data[-1] = 10
    raw = data.tobytes()
    d = ctx.load_fastq(raw)
    info = d.split()
    ref = _line_offsets_ref(raw)
    assert info.n_lines == len(ref) - 1
    assert np.array_equal(d.line_offsets(), ref)
    d.free()


STAT_FIELDS = ["base_count", "qual_count", "base_single_qual", "last_count_mismatch", "first_lcp_eq", "first_lcs_eq",
               "first_short_prefix", "first_short_suffix"]
STAT_SCALARS = ["dna_min", "dna_max", "bad_first_char", "bad_plus_record", "bad_len_record", "first_len", "last_len",
                "max_name_len", "prefix_len", "suffix_len"]


@pytest.mark.parametrize("name", CASES)
def test_analyze_matches_contract_emulation(ctx, name):
    fq, _, _ = golden_case(name)
    d = ctx.load_fastq(fq)
    d.split()
    got = d.analyze()
    want, n = emu_stats(fq)
    for f in STAT_SCALARS:
        assert getattr(got, f) == getattr(want, f), f
    for f in STAT_FIELDS:
        a, b = list(getattr(got, f)), list(getattr(want, f))
        assert a == b, "%s differs at %s" % (f, [i for i in range(len(a)) if a[i] != b[i]][:8])
    assert bytes(got.first_name[:got.first_len]) == bytes(want.first_name[:want.first_len])
    assert bytes(got.last_name[:got.last_len]) == bytes(want.last_name[:want.last_len])
    d.free()


def test_analyze_reports_malformed_records(ctx):
    good = b"@r:1\nACGT\n+\nIIII\n"
    for data, field, rec in ((good + b"@r:2\nACGT\n-\nIIII\n" + good, "bad_plus_record", 1),
                             (good + good + b"@r:3\nACG\n+\nIIII\n", "bad_len_record", 2),
                             (good + b"@r:2\nACGT\n\nIIII\n", "bad_plus_record", 1)):
        d = ctx.load_fastq(data)
        d.split()
        st = d.analyze()
        assert getattr(st, field) == rec
        d.free()


@pytest.mark.parametrize("name", CASES)
def test_qname_scan_matches_contract_emulation(ctx, name):
    from uq_b200 import host
    fq, _, _ = golden_case(name)
    st, n = emu_stats(fq)
    prefix, suffix, seps = host.derive_qname_layout(st, n)
    want, bad_w, dicts = emu_colstats(fq, len(prefix), len(suffix), seps)
    d = ctx.load_fastq(fq)
    d.split()
    got, bad_g = d.qname_scan(len(prefix), len(suffix), seps)
    assert bad_g == bad_w == -1
    for c in range(len(seps) + 1):
        for f in ("all_int", "all_canonical", "overflow", "min_len", "max_len", "n_distinct", "n_checkpoints"):
            assert getattr(got[c], f) == getattr(want[c], f), (c, f)
        if want[c].all_int:
            assert (got[c].min_val, got[c].max_val) == (want[c].min_val, want[c].max_val), c
        assert list(got[c].distinct_at) == list(want[c].distinct_at), c
        if c in dicts:
            assert d.qname_dict(c) == dicts[c], c
    d.free()


def test_qname_scan_reports_bad_separator_order(ctx):
    data = b"@a:1 x\nA\n+\nI\n@a:2 y\nA\n+\nI\n@a 3:z\nA\n+\nI\n"
    d = ctx.load_fastq(data)
    d.split()
    _, bad = d.qname_scan(2, 0, ": ")
    assert bad == 2
    d.free()


@pytest.mark.parametrize("name", CASES)
def test_pack_and_columns_match_oracle(ctx, name):
    from oracle import uq_literal as lit
    from uq_b200 import host
    fq, _, kw = golden_case(name)
    want = {}
    lit.encode(fq, stages=want, **kw)
    got = {}
    host.encode(fq, ctx=ctx, stages=got, **kw)
    assert got["dec"]["bases"] == want["dec"]["bases"] and got["dec"]["N_qual"] == want["dec"]["N_qual"]
    dna = got["dna"].download()
    qual = got["qual"].download()
    assert dna.shape == want["dna"].shape and qual.shape == want["qual"].shape
    bad = np.argwhere(dna != want["dna"])
    assert len(bad) == 0, "DNA rows differ first at %s" % bad[:4].tolist()
    bad = np.argwhere(qual != want["qual"])
    assert len(bad) == 0, "QUAL rows differ first at %s" % bad[:4].tolist()
    assert got["columns"] == want["columns"]
    for c, w, meta in zip(got["cols"], want["cols"], want["columns"]):
        assert np.array_equal(c.download(dtype=meta["dtype"]).reshape(-1), w), meta["name"]
    got["device_members"].free()


def _np_sort_unique(t):
    v = np.ascontiguousarray(t).view("V%d" % t.shape[1]).reshape(-1)
    perm = np.argsort(v, kind="stable")
    uniq, key = np.unique(v, return_inverse=True)
    return perm, key.reshape(-1), uniq.view(np.uint8).reshape(len(uniq), t.shape[1])


@pytest.mark.parametrize("n,width,alphabet", [(1, 5, 256), (2, 1, 2), (1000, 1, 3), (5000, 3, 2), (4097, 8, 2), (20000, 9, 2),
                                              (30000, 16, 2), (50000, 17, 3), (60000, 38, 2), (40000, 113, 2), (3000, 40, 256),
                                              (100000, 24, 1), (300000, 12, 4)])
def test_sort_rows_matches_numpy_stable(ctx, n, width, alphabet):
    rng = np.random.default_rng(n * 131 + width)
    t = rng.integers(0, alphabet, size=(n, width), dtype=np.uint8)
    if n > 10:
        t[rng.integers(0, n, n // 3)] = t[rng.integers(0, n, n // 3)]      # exact duplicates
        t[: n // 4, : max(width - 1, 1)] = t[0, : max(width - 1, 1)]       # long shared prefixes
    perm_w, key_w, uniq_w = _np_sort_unique(t)
    d = ctx.upload(t)
    perm, key, uniq, nu = ctx.sort_rows(d, want_perm=True, want_key=True, want_uniq=True)
    assert nu == len(uniq_w)
    assert np.array_equal(perm.download(dtype=np.uint32).reshape(-1), perm_w.astype(np.uint32))
    assert np.array_equal(key.download(dtype=np.uint32).reshape(-1), key_w.astype(np.uint32))
    assert np.array_equal(uniq.download().reshape(nu, width), uniq_w)
    g = ctx.gather_rows(d, perm)
    assert np.array_equal(g.download().reshape(n, width), t[perm_w])
    for a in (d, perm, key, uniq, g):
        a.free()


@pytest.mark.parametrize("n,width,nsplit", [(1, 9, 1), (5000, 113, 1), (70001, 38, 3), (30000, 10, 7), (9000, 4, 2), (4100, 224, 2), (3000, 3, 4),
                                           (3000, 225, 2), (2000, 788, 3), (1500, 0, 2)])
def test_streaming_partition_equals_stable_order(ctx, n, width, nsplit):
    """uqb_partition_positions / uqb_scatter_rows_segmented (multi-GPU sample sort) against numpy: pos is the inverse of
    the stable destination order, the byte buffer holds the rows of every destination in input order.  Rows the
    scatter does not take (wider than Context.SCATTER_MAX_WIDTH, or empty) are gathered through order = pos^-1."""
    rng = np.random.default_rng(n + width)
    t = rng.integers(0, 256, size=(n, width), dtype=np.uint8)
    if n > 100:
        t[: n // 3] = t[rng.integers(0, n, n // 3)]
    key = np.zeros(n, dtype=np.uint64)
    for b in range(min(8, width)):
        key |= t[:, b].astype(np.uint64) << np.uint64(8 * (7 - b))
    splits = np.sort(key[rng.integers(0, n, nsplit)])
    dest = np.searchsorted(splits, key, side="right")
    order_w = np.argsort(dest, kind="stable")
    pos_w = np.empty(n, dtype=np.uint32)
    pos_w[order_w] = np.arange(n, dtype=np.uint32)
    counts_w = np.bincount(dest, minlength=nsplit + 1)
    d = ctx.upload(t)
    pos, counts = ctx.partition_positions(d, splits)
    assert counts == counts_w.tolist()
    assert np.array_equal(pos.download(dtype=np.uint32).reshape(-1), pos_w)
    if 0 < width <= ctx.SCATTER_MAX_WIDTH:
        buf, offs = ctx.scatter_rows_segmented(d, pos, counts, 128)
    else:
        iota = ctx.upload(np.arange(n, dtype=np.uint32))
        order = ctx.scatter_u32(iota, pos)
        buf, offs = ctx.gather_rows_segmented(d, order, counts, 128)
        iota.free(); order.free()
    got = buf.download().reshape(-1)
    first = 0
    for k, c in enumerate(counts):
        assert offs[k] % 128 == 0
        seg = got[offs[k]:offs[k] + c * width].reshape(c, width)
        assert np.array_equal(seg, t[order_w[first:first + c]]), k
        first += c
    # a uint32 payload follows the same positions
    pay = ctx.upload(np.arange(n, dtype=np.uint32).view(np.uint8).reshape(n, 4))
    pbuf, poffs = ctx.scatter_rows_segmented(pay, pos, counts, 128)
    pgot = pbuf.download().reshape(-1)
    first = 0
    for k, c in enumerate(counts):
        assert np.array_equal(pgot[poffs[k]:poffs[k] + 4 * c].view(np.uint32), order_w[first:first + c].astype(np.uint32))
        first += c
    for a in (d, pos, buf, pay, pbuf):
        a.free()


@pytest.mark.parametrize("kind,n,width", [("prefix64", 30000, 113), ("staircase", 20000, 113), ("staircase", 6000, 38),
                                          ("zeros", 4000, 300), ("prefix64", 5000, 700), ("blocks", 50000, 113)])
def test_sort_rows_shared_prefixes(ctx, kind, n, width):
    """Tables whose rows agree far beyond the 8-byte round-0 key (binned qualities, right-aligned variable-length rows):
    tie groups of more than 32 differing rows go through the per-group common-prefix rounds (sort.cu)."""
    rng = np.random.default_rng(n + width)
    if kind == "prefix64":                   # four-letter alphabet, the first 64 bytes identical for all rows
        t = rng.integers(0, 4, size=(n, width), dtype=np.uint8)
        t[:, :64] = t[0, :64]
    elif kind == "staircase":                # every row differs from row 0 at one position only, positions spread over the row
        t = np.repeat(rng.integers(0, 4, size=(1, width), dtype=np.uint8), n, axis=0)
        pos = 8 + (np.arange(n) % (width - 8))
        t[np.arange(n), pos] = rng.integers(4, 9, size=n).astype(np.uint8)
    elif kind == "blocks":                   # 200 distinct 40-byte prefixes, each followed by one of a few tails
        pre = rng.integers(0, 4, size=(200, 40), dtype=np.uint8)
        tails = rng.integers(0, 4, size=(37, width - 40), dtype=np.uint8)
        t = np.concatenate([pre[rng.integers(0, 200, n)], tails[rng.integers(0, 37, n)]], axis=1)
    else:                                    # right-aligned rows: many leading zero bytes, a few significant bytes
        t = np.zeros((n, width), dtype=np.uint8)
        sig = rng.integers(1, 40, size=n)
        for i in range(n):
            t[i, width - sig[i]:] = rng.integers(1, 3, size=sig[i])
    perm_w, key_w, uniq_w = _np_sort_unique(t)
    d = ctx.upload(t)
    perm, key, uniq, nu = ctx.sort_rows(d, want_perm=True, want_key=True, want_uniq=True)
    assert nu == len(uniq_w)
    assert np.array_equal(perm.download(dtype=np.uint32).reshape(-1), perm_w.astype(np.uint32))
    assert np.array_equal(key.download(dtype=np.uint32).reshape(-1), key_w.astype(np.uint32))
    assert np.array_equal(uniq.download().reshape(nu, width), uniq_w)
    for a in (d, perm, key, uniq):
        a.free()


@pytest.mark.parametrize("n,width", [(1, 1), (1, 7), (9, 1), (65, 64), (64, 65), (1000, 38), (777, 113), (5, 300), (130, 129),
                                     (1001, 5001), (300, 1000), (3, 17501), (513, 200), (259, 257)])
def test_layouts_match_numpy(ctx, n, width):
    from oracle.uq_literal import PATTERNS, apply_pattern
    rng = np.random.default_rng(n + 7 * width)
    t = rng.integers(0, 256, size=(n, width), dtype=np.uint8)
    d = ctx.upload(t)
    for p in PATTERNS:
        want = np.frombuffer(apply_pattern(t, p).tobytes(order="A"), dtype=np.uint8)
        s = ctx.layout(d, p)
        got = s.download().reshape(-1)
        assert np.array_equal(got, want), p
        back = ctx.unlayout(s, n, width, p)
        assert np.array_equal(back.download().reshape(n, width), t), p
        s.free(); back.free()
    d.free()


@pytest.mark.parametrize("name", CASES)
def test_encode_matches_reference_container(ctx, name):
    from oracle import uq_literal as lit
    from uq_b200 import host
    fq, uq, kw = golden_case(name)
    want_members, want_cfg = lit.read_container(uq)
    got_members, got_cfg = host.encode(fq, ctx=ctx, **kw)
    assert_members_equal(got_members, want_members, name)
    assert_config_equal(got_cfg, want_cfg, name)


@pytest.mark.parametrize("name", CASES)
def test_decode_of_reference_container(ctx, name):
    from oracle import uq_literal as lit
    from uq_b200 import host
    fq, uq, kw = golden_case(name)
    members, cfg = lit.read_container(uq)
    out = host.decode(members, cfg, ctx=ctx).tobytes()
    if kw["sort"] in (None, "None"):
        assert out == fq
    else:
        assert records_multiset(out) == records_multiset(fq)


@pytest.mark.parametrize("kind,length", [("illumina", 100), ("genome", 150), ("casava", 100), ("ont", (50, 3000))])
def test_device_synth_equals_host_synth(ctx, kind, length):
    from oracle import synth
    n, first = 300, 12345
    kw = dict(kind=kind, n=n, length=length, seed=77, first=first)
    dev_kw = {}
    if kind == "genome":
        kw.update(genome=5000, pool=40)
        dev_kw.update(genome=5000, pool=40)
    if kind == "ont":
        dev_kw.update(len_table=synth.ont_length_table(*length))
    want = synth.make_fastq(**kw)
    got = ctx.synth(kind, n, length, 77, first=first, **dev_kw)
    data = got.download().tobytes()
    assert len(data) == len(want)
    assert data == want
    got.free()


def _roundtrip(ctx, dev_bytes, **kw):
    """encode on the device, write nothing to disk, decode on the device."""
    from uq_b200 import host
    fq = ctx.adopt_fastq(dev_bytes)
    members, cfg = host.encode_device(ctx, fq, **kw)
    host_members = members.download()
    members.free()
    fq.free()
    return host_members, cfg, host.decode(host_members, cfg, ctx=ctx)


def test_roundtrip_1m_reads_unsorted_is_byte_exact(ctx):
    dev = ctx.synth("illumina", 1_000_000, 100, 1001)
    original = dev.download().copy()
    members, cfg, out = _roundtrip(ctx, dev, sort="None", raw=["DNA", "QUAL", "QNAME"], pattern=["0.1", "0.1"])
    assert cfg["bits_per_base"] == 2 and cfg["bits_per_quality"] == 6 and cfg["N_qual"] == {"N": 0}
    assert members["DNA.raw"].shape == (1_000_000, 25) and members["QUAL.raw"].shape == (1_000_000, 75)
    assert [c["dtype"] for c in cfg["QNAME_columns"]] == ["uint8", "uint16", "uint16", "uint32"]
    assert out.tobytes() == original.tobytes()
    dev.free()


def test_roundtrip_sorted_keyed_is_a_sorted_permutation(ctx):
    n = 400_000
    dev = ctx.synth("genome", n, 150, 1002, genome=40_000, pool=50_000)
    original = dev.download().tobytes()
    members, cfg, out = _roundtrip(ctx, dev, sort="DNA")
    assert records_multiset(out.tobytes()) == records_multiset(original)
    key = members["DNA.key"]
    assert np.all(np.diff(key.astype(np.int64)) >= 0), "sorted-on key must be non-decreasing"
    u = members["DNA"]
    v = np.ascontiguousarray(u).view("V%d" % u.shape[1]).reshape(-1)
    assert np.array_equal(np.sort(v), v) and len(np.unique(v)) == len(v), "unique table must be strictly ascending"
    # stable: within equal DNA, records keep file order -> QNAME-less check through decode order of duplicates
    dev.free()


def test_roundtrip_variable_length_sort_qual(ctx):
    from oracle import synth
    n = 3000
    tab = synth.ont_length_table(1000, 20000)
    dev = ctx.synth("ont", n, (1000, 20000), 1005, len_table=tab)
    original = dev.download().tobytes()
    members, cfg, out = _roundtrip(ctx, dev, sort="QUAL")
    assert cfg["variable_read_lengths"] is True and cfg["bits_per_quality"] == 7
    assert records_multiset(out.tobytes()) == records_multiset(original)
    dev.free()


@pytest.mark.parametrize("sort", ["None", "QUAL"])
def test_long_variable_reads_equal_the_literal_oracle(ctx, sort):
    """Reads of 64 .. 3 000 bases (too long for record tiles: direct histogram, one-CTA-per-read packer, leading-zero
    aware sort) against the pinned literal oracle, member by member."""
    from oracle import synth, uq_literal as lit
    from uq_b200 import host
    tab = synth.ont_length_table(64, 3000)
    dev = ctx.synth("ont", 120, (64, 3000), 77, len_table=tab)
    fastq = dev.download().tobytes()
    dev.free()
    kw = dict(sort=sort) if sort != "None" else dict(sort="None", raw=["DNA", "QUAL", "QNAME"])
    want, want_cfg = lit.encode(fastq, **kw)
    got, got_cfg = host.encode(fastq, ctx=ctx, **kw)
    assert want_cfg["variable_read_lengths"] is True
    assert_members_equal(got, want)
    assert_config_equal(got_cfg, want_cfg)
    assert host.decode(got, got_cfg, ctx=ctx).tobytes() == lit.decode(want, want_cfg)


def test_streamed_load_and_async_download_match_the_serial_path(ctx):
    """uqb_fastq_load_streamed (chunked H2D overlapped with split + Pass-1 statistics) and the asynchronous
    member downloads must give exactly the arrays of the serial path."""
    from uq_b200 import host
    from emu import emu_stats
    dev = ctx.synth("genome", 300_000, 150, 77, genome=30_000, pool=50_000)
    data = dev.download().copy()
    dev.free()
    want, want_cfg = host.encode(data, ctx=ctx, sort="DNA")
    pin = ctx.pinned_empty(data.size)
    pin.array[:] = data
    for chunk in (1 << 20, 3 * 16384, 0):
        fq = ctx.load_fastq_streamed(pin, chunk_bytes=chunk)
        info = fq.split()
        assert info.n_reads == 300_000 and info.status == 0
        bufs = {}
        def sink(name, nbytes):
            bufs[name] = ctx.pinned_empty(nbytes)
            return bufs[name].array
        members, cfg = host.encode_device(ctx, fq, sort="DNA", sink=sink)
        got = members.download()
        assert_members_equal(got, want, "streamed chunk=%d" % chunk)
        assert_config_equal(cfg, want_cfg)
        members.free()
        fq.free()
        for b in bufs.values():
            b.free()
    # statistics of a streamed handle equal the contract emulation (small case, tiny chunks)
    fq_small, _, _ = golden_case("c3_casava_raw")
    pin2 = ctx.pinned_empty(len(fq_small))
    pin2.array[:] = np.frombuffer(fq_small, dtype=np.uint8)
    h = ctx.load_fastq_streamed(pin2, chunk_bytes=16384)
    h.split()
    st = h.analyze()
    ref, _ = emu_stats(fq_small)
    for f in STAT_SCALARS:
        assert getattr(st, f) == getattr(ref, f), f
    for f in STAT_FIELDS:
        assert list(getattr(st, f)) == list(getattr(ref, f)), f
    h.free(); pin2.free(); pin.free()


def test_ntrick_new_quality_branch_encodes_like_the_reference_and_decodes(ctx):
    """Q3: the reference encodes such a file (N gets quality code len(qualities)+1) but cannot decode it and stores
    the original quality nowhere.  The arrays and the reference's config keys must stay bit-exact; the extra
    N_qual_symbol key makes the container decodable here - byte for byte."""
    from oracle import uq_literal as lit
    from uq_b200 import host
    from conftest import hiseq_like_fastq
    fq = hiseq_like_fastq()
    for kw in (dict(sort="None", raw=["DNA", "QUAL", "QNAME"]), dict(sort="QUAL")):
        want, want_cfg = lit.encode(fq, **kw)
        got, got_cfg = host.encode(fq, ctx=ctx, **kw)
        assert want_cfg["N_qual"] == {"N": len(want_cfg["qualities"]) + 1}         # the branch fired
        assert_members_equal(got, want)
        extra = dict(got_cfg)
        assert extra.pop("N_qual_symbol") == {"N": "#"}
        assert_config_equal(extra, want_cfg)
        text = host.decode(got, got_cfg, ctx=ctx).tobytes()
        if kw["sort"] == "None":
            assert text == fq
        else:
            assert records_multiset(text) == records_multiset(fq)
        stripped = {k: v for k, v in got_cfg.items() if k != "N_qual_symbol"}      # a reference-written container
        with pytest.raises(host.UQError, match="no quality symbol"):
            host.decode(got, stripped, ctx=ctx)


@pytest.mark.parametrize("name", ["c2_keyed_sortDNA", "c3_casava_sortQNAME", "c5_variable_sortQUAL"])
def test_mix_feed_serves_every_mix_like_a_fresh_encode(ctx, name):
    """SURVEY 8(f1): the --test feed loads and packs once, sorts each table at most once and serves every member of
    every (sort, raw, pattern) mix as a gather / layout of resident arrays - the members must be those of a fresh
    encode with the same options, bit for bit (dtype, shape, memory order)."""
    from uq_b200 import host
    fq, _, kw = golden_case(name)
    dfq = ctx.load_fastq(fq)
    feed = host.MixFeed(ctx, dfq, pad=kw["pad"], notricks=kw["notricks"])
    launches_before = ctx.launches
    pats = ['0.1', '1.1', '2.1', '3.1', '0.2', '1.2', '2.2', '3.2']
    raws = [('DNA', 'QUAL', 'QNAME'), ('DNA', 'QUAL'), ('QUAL', 'QNAME'), ('DNA', 'QNAME'), ('DNA',), ('QUAL',), ('QNAME',), (None,)]
    n = 0
    for i, raw in enumerate(raws):
        for j, sort in enumerate(['DNA', 'QUAL', 'QNAME', None]):
            pat = [pats[(i + j) % 8], pats[(3 * i + j + 5) % 8]]
            opts = dict(sort=sort if sort else 'None', raw=[r if r else 'none' for r in raw], pattern=pat)
            got = feed.members(**opts)
            want, want_cfg = host.encode(fq, ctx=ctx, pad=kw["pad"], notricks=kw["notricks"], **opts)
            assert_members_equal(got, want, "%s %r" % (name, opts))
            assert_config_equal(feed.config(**opts), want_cfg)
            n += 1
    assert n == 32
    # the whole sweep cost three sorts: asking again launches nothing
    before = ctx.launches
    feed.members(sort='QUAL', raw=['DNA'], pattern=['2.2', '1.1'])
    feed.members(sort='QUAL', raw=['DNA'], pattern=['2.2', '1.1'])
    assert ctx.launches - before <= 40
    feed.free()
    dfq.free()


def test_encode_reports_malformed_record_by_entry(ctx):
    """host.encode names the record of a third line without '+' and of a quality line shorter than its sequence."""
    from uq_b200 import host
    dev = ctx.synth("genome", 700_000, 150, 77, genome=70_000, pool=100_000)
    data = dev.download().copy()
    dev.free()
    lines = data[:400_000].tobytes().split(b"\n")
    lines[4 * 700 + 2] = b"-"                               # record 700: third line does not start with '+'
    lines[4 * 900 + 3] = lines[4 * 900 + 3][:-3]            # record 900: quality line three symbols short
    broken = b"\n".join(lines[:4 * 1000]) + b"\n"
    with pytest.raises(host.UQError, match="entry 700 the third line"):
        host.encode(broken, ctx=ctx)
    lines[4 * 700 + 2] = b"+"
    broken = b"\n".join(lines[:4 * 1000]) + b"\n"
    with pytest.raises(host.UQError, match="for entry 901"):
        host.encode(broken, ctx=ctx)
