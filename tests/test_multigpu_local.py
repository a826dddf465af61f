"""The sharded (one container from W ranks) encode and decode on ONE GPU: W emulated ranks (host threads, one context
each, uq_b200.multigpu.LocalComm) run exactly the code the NCCL ranks run - merged statistics, partition-first sample
sort (uqb_partition_positions, uqb_scatter_rows_segmented / uqb_gather_rows_segmented, uqb_compact_segments,
uqb_scatter_u32), global order, per-rank layouts and their placement, sharded decode - and the result must equal the
single-GPU encode of the whole file member by member.  SURVEY section 4(d) / 8(e)."""
import json

import numpy as np
import pytest

from conftest import assert_members_equal, records_multiset

pytestmark = pytest.mark.gpu

PATTERNS = ['0.1', '1.1', '2.1', '3.1', '0.2', '1.2', '2.2', '3.2']

# (kind, reads, read length, options)
CASES = [
    ("genome", 24000, 60, dict(sort="DNA")),
    ("genome", 24000, 60, dict(sort="None", raw=["DNA", "QUAL", "QNAME"])),
    ("genome", 9000, 40, dict(sort="QUAL", raw=["DNA"])),
    ("casava", 26000, 50, dict(sort="QNAME")),
    ("casava", 8000, 50, dict(sort="DNA", raw=["QNAME", "QUAL"])),
    ("illumina", 7000, 30, dict()),
    ("genome", 9000, 40, dict(sort="DNA", pattern=["2.2", "1.1"])),
    ("genome", 9000, 40, dict(sort="QNAME", raw=["QUAL"], pattern=["3.1", "3.2"])),
    # variable-length reads of up to 900 bases: DNA and QUAL rows wider than Context.SCATTER_MAX_WIDTH
    ("ont", 6000, (50, 900), dict(sort="QUAL")),
    ("ont", 6000, (50, 900), dict(sort="QNAME", raw=["DNA", "QUAL"])),
]


def _cuts(n, world):
    """uneven contiguous ranges; rank 0 is the largest (it must hold the first 10001 reads)"""
    wts = [0.55, 0.45] if world == 2 else [0.46] + [0.54 / (world - 1)] * (world - 1)
    return [0] + [int(n * sum(wts[:k + 1])) for k in range(world - 1)] + [n]


def _gen(kind, n, length, first=0):
    from oracle import synth
    kwg = dict(genome=max(4 * length, 4000), pool=max(1, 3500)) if kind == "genome" else {}
    return synth.make_fastq(kind=kind, n=n, length=length, seed=21, first=first, **kwg)


def _sharded_encode(world, whole_records, kw, merge=False, window=0):
    """whole_records: list of per-record byte strings -> (members on rank 0, config).  window > 0: the row exchanges go
    through a peer window of that many bytes (direct stores into the other ranks' memory)."""
    import os
    from uq_b200 import multigpu as mg
    cuts = _cuts(len(whole_records), world)

    def body(ctx, comm):
        os.environ["UQB_MG_MERGE"] = "1" if merge else "0"
        if window:
            comm.open_window(ctx, window)
        shard = b"".join(whole_records[cuts[comm.rank]:cuts[comm.rank + 1]])
        fq = ctx.load_fastq(shard)
        res, cfg = mg.encode_sharded(ctx, comm, fq, **kw)
        members = mg.assemble(comm, res)
        res.free(); fq.free()
        return members, cfg

    try:
        out = mg.run_local(world, body)
    finally:
        os.environ["UQB_MG_MERGE"] = "0"
    cfgs = [json.dumps(c, sort_keys=True, default=str) for _, c in out]
    assert len(set(cfgs)) == 1                          # the config is identical on every rank
    return out[0]


def _records(fq):
    ls = fq.split(b"\n")[:-1]
    return [b"\n".join(ls[i:i + 4]) + b"\n" for i in range(0, len(ls), 4)]


@pytest.fixture(scope="module")
def ctx():
    from uq_b200.device import Context
    c = Context(0)
    yield c
    c.close()


@pytest.mark.parametrize("world", [2, 3, 4])
@pytest.mark.parametrize("case", range(len(CASES)))
def test_sharded_encode_equals_single_gpu(ctx, world, case):
    from uq_b200 import host
    kind, n, length, kw = CASES[case]
    whole = _gen(kind, n, length)
    want, want_cfg = host.encode(whole, ctx=ctx, **kw)
    got, cfg = _sharded_encode(world, _records(whole), kw)
    assert_members_equal(got, want, "%s world=%d %r" % (kind, world, kw))
    assert json.loads(json.dumps(cfg, default=str)) == json.loads(json.dumps(want_cfg, default=str))


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("case", range(len(CASES)))
def test_sharded_encode_through_peer_window(ctx, world, case):
    """the device-initiated exchange (uqb_scatter_rows_to into the peers' receive slots, barriers around it) gives the
    same container; the window is small enough that the largest table of some cases falls back to the collective"""
    from uq_b200 import host
    kind, n, length, kw = CASES[case]
    whole = _gen(kind, n, length)
    want, _ = host.encode(whole, ctx=ctx, **kw)
    got, _ = _sharded_encode(world, _records(whole), kw, window=3 * 600_000)
    assert_members_equal(got, want, "window %s world=%d %r" % (kind, world, kw))


@pytest.mark.parametrize("case", [0, 2, 3, 8, 9])
def test_sharded_encode_merge_variant(ctx, case):
    """the skew-proof variant (local sort first, only locally unique rows travel) gives the same container"""
    from uq_b200 import host
    kind, n, length, kw = CASES[case]
    whole = _gen(kind, n, length)
    want, _ = host.encode(whole, ctx=ctx, **kw)
    got, _ = _sharded_encode(2, _records(whole), kw, merge=True)
    assert_members_equal(got, want, "merge %s %r" % (kind, kw))


@pytest.mark.parametrize("pattern", PATTERNS)
def test_sharded_layouts_all_patterns(ctx, pattern):
    """every --pattern, keyed and raw, over 3 ranks: per-rank layout + placement = the single-GPU stream"""
    from uq_b200 import host
    whole = _gen("genome", 6000, 37)
    other = PATTERNS[(PATTERNS.index(pattern) + 3) % 8]
    for kw in (dict(sort="QUAL", pattern=[pattern, other]), dict(sort="None", raw=["DNA", "QUAL"], pattern=[other, pattern])):
        want, _ = host.encode(whole, ctx=ctx, **kw)
        got, _ = _sharded_encode(3, _records(whole), kw)
        assert_members_equal(got, want, "pattern %s %r" % (pattern, kw))


def test_sharded_skewed_table_takes_the_merge_route(ctx):
    """a table of (almost) identical rows fools the sample: one rank would receive everything -> merge variant"""
    from uq_b200 import host
    recs = [b"@r:%d:%d\nACGTACGTACGTACGTACGT\n+\nIIIIIIIIIIIIIIIIIIII\n" % (i % 7, i) for i in range(9000)]
    recs[5] = b"@r:5:5\nTTTTACGTACGTACGTACGA\n+\nIIIIIIIIIIIIIIIIIII#\n"
    whole = b"".join(recs)
    for kw in (dict(sort="DNA"), dict(sort="QUAL", raw=["QNAME"])):
        want, _ = host.encode(whole, ctx=ctx, **kw)
        got, _ = _sharded_encode(2, recs, kw)
        assert_members_equal(got, want, "skew %r" % (kw,))


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("kw", [dict(sort="DNA"), dict(sort="None", raw=["DNA", "QUAL", "QNAME"], pattern=["1.1", "2.2"]),
                                dict(sort="QNAME", raw=["QUAL"], pattern=["3.2", "0.2"]), dict(pattern=["2.1", "3.1"])])
def test_sharded_decode_round_trip(ctx, world, kw):
    """container written by the single-GPU encode -> W ranks decode contiguous record ranges -> concatenated text.
    Unsorted containers must reproduce the file byte for byte; sorted ones the same records in the container's order
    (= what the single-GPU decode emits)."""
    from uq_b200 import host, multigpu as mg
    whole = _gen("casava", 9000, 45)
    members, cfg = host.encode(whole, ctx=ctx, **kw)
    single = host.decode(members, cfg, ctx=ctx).tobytes()

    def body(c, comm):
        data, a, b = mg.decode_sharded(c, comm, members, cfg)
        return bytes(data), a, b

    parts = mg.run_local(world, body)
    assert [p[1] for p in parts] == [0] + [p[2] for p in parts[:-1]] and parts[-1][2] == 9000
    text = b"".join(p[0] for p in parts)
    assert text == single
    if kw.get("sort") in (None, "None"):
        assert text == whole
    else:
        assert records_multiset(text) == records_multiset(whole)


def test_sharded_variable_length_encode_and_decode(ctx):
    from oracle import synth
    from uq_b200 import host, multigpu as mg
    whole = synth.make_fastq(kind="ont", n=600, length=(50, 900), seed=8)
    kw = dict(sort="QUAL", pattern=["0.2", "2.1"])
    want, want_cfg = host.encode(whole, ctx=ctx, **kw)
    got, cfg = _sharded_encode(2, _records(whole), kw)
    assert_members_equal(got, want, "variable length")
    parts = mg.run_local(2, lambda c, comm: bytes(mg.decode_sharded(c, comm, got, cfg)[0]))
    assert records_multiset(b"".join(parts)) == records_multiset(whole)


def test_local_comm_collectives(ctx):
    """the emulated collectives themselves: object all-gather, row all-to-all, all-gather of uneven row blocks"""
    from uq_b200 import multigpu as mg
    world, w = 3, 5

    def body(c, comm):
        r = comm.rank
        assert comm.all_gather_object(("x", r)) == [("x", k) for k in range(world)]
        send_counts = [r + 1, 2, 3]                                  # rows to rank 0, 1, 2 (6, 7, 8 rows per rank)
        rows = np.arange(sum(send_counts) * w, dtype=np.uint8).reshape(-1, w) + 40 * r
        recv_counts = comm.exchange_counts(send_counts)
        d = c.upload(rows)
        got = comm.all_to_all_rows(c, d, send_counts, recv_counts).download().reshape(-1, w)
        full = comm.all_gather_rows(c, d, [6, 7, 8]).download().reshape(-1, w)
        return rows, send_counts, got, full

    out = mg.run_local(world, body)
    for r in range(world):
        want = []
        for src in range(world):
            rows, sc, _, _ = out[src]
            off = sum(sc[:r])
            want.append(rows[off:off + sc[r]])
        assert np.array_equal(out[r][2], np.concatenate(want))
        assert np.array_equal(out[r][3], np.concatenate([out[k][0] for k in range(world)]))


def test_malformed_container_is_refused_not_faulted(ctx):
    """a key that points outside its unique table, or a variable-length row without a valid marker, must raise"""
    from oracle import synth
    from uq_b200 import host
    whole = _gen("genome", 3000, 40)
    members, cfg = host.encode(whole, ctx=ctx, sort="DNA")
    bad = dict(members)
    k = members["DNA.key"].copy()
    k[17] = members["DNA"].shape[0] + 5 if k.dtype.itemsize > 1 else 255
    if int(k[17]) < members["DNA"].shape[0]:
        pytest.skip("unique table too large for an out-of-range uint8 key")
    bad["DNA.key"] = k
    with pytest.raises(host.UQError, match="points outside"):
        host.decode(bad, cfg, ctx=ctx)
    vfq = synth.make_fastq(kind="ont", n=50, length=(30, 200), seed=3)
    vm, vcfg = host.encode(vfq, ctx=ctx, sort="None", raw=["DNA", "QUAL", "QNAME"])
    vbad = dict(vm)
    t = vm["DNA.raw"].copy()
    assert host.decode(vm, vcfg, ctx=ctx).tobytes() == vfq
    if 8 * t.shape[1] - vcfg["bits_per_base"] * (vcfg["dna_max"] + 1) >= 1:      # there are pad bits in front of the widest marker
        t[7, 0] |= 0x80
        vbad["DNA.raw"] = t
        from uq_b200.device import DeviceError
        with pytest.raises(DeviceError, match="marker"):
            host.decode(vbad, vcfg, ctx=ctx)
