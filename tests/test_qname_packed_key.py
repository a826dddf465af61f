"""QNAME tables sorted on one packed 64-bit key (host.qname_key_plan): the plan on hand-written column lists without a
GPU; on the GPU, the packed-key sort against the sort of the big-endian rows it replaces (perm, key, key_sorted, unique
count and unique columns), and whole encodes against the row path."""
import numpy as np
import pytest

from conftest import assert_config_equal, assert_members_equal


def ints(lo, hi, dtype, offset=False):
    return {'format': 'integers', 'min': lo, 'max': hi, 'dtype': dtype, 'offset': offset}


def mapping(k):
    return {'format': 'mapping', 'map': ['t%03d' % i for i in range(k)], 'dtype': 'uint8' if k <= 255 else 'uint16'}


def strings(w):
    return {'format': 'strings', 'longest': w, 'dtype': '|S%d' % w}


BENCH = [ints(1, 8, 'uint8'), ints(1101, 2678, 'uint16'), ints(1002, 29996, 'uint16'), ints(1006, 199987, 'uint32')]


# ------------------------------------------------------------------------------------------------
# plan (CPU)
# ------------------------------------------------------------------------------------------------
def test_plan_of_bench_names_is_47_bits_in_column_order():
    from uq_b200.host import qname_key_plan
    plan = qname_key_plan(BENCH)
    assert plan == [(44, 3, 1), (33, 11, 1101), (18, 15, 1002), (0, 18, 1006)]
    assert sum(b for _, b, _ in plan) == 47


def test_plan_constant_offset_and_mapping_columns():
    from uq_b200.host import qname_key_plan
    plan = qname_key_plan([ints(7, 7, 'uint8'), ints(-5, 10, 'uint8', offset=True), mapping(1), mapping(2), ints(0, 300, 'uint16')])
    assert plan == [(14, 0, 7), (10, 4, 0), (10, 0, 0), (9, 1, 0), (0, 9, 0)]


def test_plan_of_64_bits_and_of_65_bits():
    from uq_b200.host import qname_key_plan
    plan = qname_key_plan([ints(0, 2 ** 40 - 1, 'uint64'), ints(5, 5 + 2 ** 24 - 1, 'uint32')])
    assert plan == [(24, 40, 0), (0, 24, 5)]
    assert qname_key_plan([ints(0, 2 ** 40 - 1, 'uint64'), ints(5, 5 + 2 ** 24, 'uint32')]) is None
    assert qname_key_plan([ints(0, 2 ** 64 - 1, 'uint64')]) == [(0, 64, 0)]


def test_plan_with_a_strings_column_is_none():
    from uq_b200.host import qname_key_plan
    assert qname_key_plan(BENCH[:2] + [strings(6)]) is None


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    from uq_b200.device import Context
    c = Context(0)
    yield c
    c.close()


def _values(rng, meta, n, unique=False):
    """encoded column values: integers as stored (value, or value - min for an offset column), mapping ranks"""
    dt = np.dtype(meta['dtype'])
    if meta['format'] == 'mapping':
        return rng.integers(0, len(meta['map']), n).astype(dt)
    lo, hi = (0, meta['max'] - meta['min']) if meta['offset'] else (meta['min'], meta['max'])
    if unique:
        return (lo + rng.permutation(n).astype(np.uint64)).astype(dt)
    v = rng.integers(0, hi - lo, n, dtype=np.uint64, endpoint=True) + np.uint64(lo)
    v[:2] = [lo, hi]
    return v.astype(dt)


LAYOUTS = {
    "bench": (BENCH, False),
    "duplicates": ([ints(1, 4, 'uint8'), mapping(3), ints(10, 40, 'uint8'), ints(9, 9, 'uint16')], False),
    "all_unique": ([ints(1, 8, 'uint8'), ints(0, 2 ** 22, 'uint32')], True),
    "64_bits": ([ints(-2 ** 30, 2 ** 30 - 1, 'uint32', offset=True), mapping(7), ints(0, 2 ** 30 - 1, 'uint64')], False),
}


@pytest.mark.gpu
@pytest.mark.parametrize("n", [5000, (1 << 20) + 70001])
@pytest.mark.parametrize("layout", sorted(LAYOUTS))
def test_packed_key_sort_equals_row_sort(ctx, layout, n):
    from uq_b200 import host
    columns, unique = LAYOUTS[layout]
    plan = host.qname_key_plan(columns)
    assert plan is not None and (layout != "64_bits" or sum(b for _, b, _ in plan) == 64)
    rng = np.random.default_rng(n)
    host_cols = [_values(rng, m, n, unique=unique and m is columns[-1]) for m in columns]
    cols = [ctx.upload(c) for c in host_cols]
    rows = host.qname_rows(ctx, cols, columns)
    table = ctx.columns_to_key(cols, plan)
    res = []
    for t in (rows, table):
        perm, key, uniq, nu, ks = ctx.sort_rows(t, want_perm=True, want_key=True, want_uniq=True, want_key_sorted=True)
        ucols = host.qname_columns(ctx, uniq, columns, None if t is rows else plan)
        res.append([a.download(dtype=np.uint32).reshape(-1) for a in (perm, key, ks)] + [nu] +
                   [u.download(dtype=np.dtype(m['dtype'])).reshape(-1) for u, m in zip(ucols, columns)])
        for a in [perm, key, uniq, ks] + ucols:
            a.free()
    rows.free(); table.free()
    for c in cols:
        c.free()
    want, got = res
    for i, name in enumerate(["perm", "key", "key_sorted", "n_unique"] + [m['format'] for m in columns]):
        assert np.array_equal(got[i], want[i]), "%s n=%d: %s differs" % (layout, n, name)
    # and the row sort itself is numpy's stable lexicographic order
    order = np.lexsort(host_cols[::-1])
    assert np.array_equal(want[0], order)
    assert want[3] == (n if unique else len(np.unique(np.stack(host_cols, 1).astype(np.uint64), axis=0)))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["genome", "casava"])
@pytest.mark.parametrize("mix", [dict(sort="DNA"), dict(sort="QNAME"), dict(sort="QNAME", raw=["QNAME"]), dict(sort="None")])
def test_encode_with_packed_key_equals_row_path(ctx, kind, mix, monkeypatch):
    from uq_b200 import host
    extra = dict(genome=200_000, pool=40_000) if kind == "genome" else {}
    fq = ctx.synth(kind, 200_000, 60, 11, **extra).download().tobytes()
    got, cfg = host.encode(fq, ctx=ctx, **mix)
    assert host.qname_key_plan(cfg['QNAME_columns']) is not None
    monkeypatch.setattr(host, "qname_key_plan", lambda columns: None)
    want, want_cfg = host.encode(fq, ctx=ctx, **mix)
    assert_members_equal(got, want, "%s %r" % (kind, mix))
    assert_config_equal(cfg, want_cfg, "%s %r" % (kind, mix))
