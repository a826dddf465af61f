"""Round-0 row sort at sizes that take the MSD bucket path of uqb_radix_sort (n >= 2^20 keys): every case is checked
against a stable numpy sort, and every case holds both buckets that one CTA finishes in shared memory and buckets too
large for one CTA (split again by the next 8 bits, or cut into runs of equal keys)."""
import numpy as np
import pytest

from oracle.synth import rnd, _skew, ST_GENOME, ST_NPOS, ST_OFF, ST_POOL, ST_QA, ST_QB, ST_SUB, ST_SUBV

pytestmark = pytest.mark.gpu

MSD_MIN_N = 1 << 20
TILE = 4096


@pytest.fixture(scope="module")
def ctx():
    from uq_b200.device import Context
    c = Context(0)
    yield c
    c.close()


def _be_words(t):
    n, w = t.shape
    pad = np.zeros((n, -(-w // 8) * 8), dtype=np.uint8)
    pad[:, :w] = t
    return [pad[:, i:i + 8].copy().view(">u8").reshape(-1) for i in range(0, pad.shape[1], 8)]


def _np_sort_unique(t):
    """numpy argsort(kind='stable') + unique(return_inverse) of the rows, through big-endian words and lexsort."""
    words = _be_words(t)
    perm = np.lexsort(words[::-1])                  # stable, first word major
    head = np.zeros(len(perm), dtype=bool)
    head[0] = True
    for c in words:
        s = c[perm]
        head[1:] |= s[1:] != s[:-1]
    gid = np.cumsum(head, dtype=np.int64) - 1
    key = np.empty(len(perm), dtype=np.int64)
    key[perm] = gid
    return perm, key, gid, t[perm[head]]


def _check(ctx, t):
    assert len(t) >= MSD_MIN_N
    perm_w, key_w, ks_w, uniq_w = _np_sort_unique(t)
    d = ctx.upload(np.ascontiguousarray(t))
    perm, key, uniq, nu, ks = ctx.sort_rows(d, want_perm=True, want_key=True, want_uniq=True, want_key_sorted=True)
    assert nu == len(uniq_w)
    assert np.array_equal(perm.download(dtype=np.uint32).reshape(-1), perm_w.astype(np.uint32))
    assert np.array_equal(key.download(dtype=np.uint32).reshape(-1), key_w.astype(np.uint32))
    assert np.array_equal(ks.download(dtype=np.uint32).reshape(-1), ks_w.astype(np.uint32))
    assert np.array_equal(uniq.download().reshape(nu, t.shape[1]), uniq_w)
    for a in (d, perm, key, uniq, ks):
        a.free()


def _rows_from_keys(key0, tail):
    """rows = be64(key0) followed by the bytes of `tail` (uint8[n][k])."""
    head = key0.astype(">u8").view(np.uint8).reshape(-1, 8)
    return np.concatenate([head, tail], axis=1)


def _bench_keys(n, seed=1002, length=150):
    """First 8 bytes of the bench's packed DNA (2-bit bases) and QUAL (6-bit symbols) rows, configs[1] duplication scaled to
    n reads (genome of n / 10 positions, quality pool of n / 5 strings), and the pool / genome index of every read."""
    r = np.arange(n, dtype=np.uint64)
    off = rnd(seed, ST_OFF, r) % np.uint64(max(n // 10, 1000))
    pidx = rnd(seed, ST_POOL, r) % np.uint64(max(n // 5, 1))
    alpha = np.array([35] + list(range(37, 75)))
    dna = np.zeros(n, np.uint64)
    qual = np.zeros(n, np.uint64)
    with np.errstate(over="ignore"):
        for p in range(30):
            pos = np.uint64(p)
            gidx = r * np.uint64(1 << 20) + pos
            b = (rnd(seed, ST_GENOME, off + pos) & np.uint64(3)).astype(np.int64)
            sub = (rnd(seed, ST_SUB, gidx) % np.uint64(1000)) == 0
            b = np.where(sub, (b + 1 + (rnd(seed, ST_SUBV, gidx) % np.uint64(3)).astype(np.int64)) & 3, b)
            isn = (rnd(seed, ST_NPOS, gidx) % np.uint64(200)) == 0
            dna = (dna << np.uint64(2)) | np.where(isn, 0, b).astype(np.uint64)
            if p < 10:
                qi = pidx * np.uint64(length) + pos
                q = np.where(isn, 35, 74 - _skew(rnd(seed, ST_QA, qi), rnd(seed, ST_QB, qi), 38))
                qual = (qual << np.uint64(6)) | np.searchsorted(alpha, q).astype(np.uint64)
    return dna, qual, off, pidx


def _tail(idx, k=8):
    """k bytes that are a function of idx: rows with the same idx are identical."""
    return (rnd(77, 1, idx.astype(np.uint64))[:, None] >> (np.arange(k, dtype=np.uint64) * np.uint64(8))).astype(np.uint8)


def test_uniform_random_rows(ctx):
    rng = np.random.default_rng(1)
    n = 3 * MSD_MIN_N + 77
    t = rng.integers(0, 256, size=(n, 16), dtype=np.uint8)
    t[rng.integers(0, n, 20000)] = t[5]                 # one key far over a CTA's capacity
    _check(ctx, t)


def test_uniform_random_keys_width8(ctx):
    rng = np.random.default_rng(2)
    n = MSD_MIN_N + 12345
    t = rng.integers(0, 256, size=(n, 8), dtype=np.uint8)
    t[rng.integers(0, n, n // 4)] = t[rng.integers(0, n, n // 4)]
    _check(ctx, t)


@pytest.fixture(scope="module")
def bench_keys():
    return _bench_keys(5_000_000)


@pytest.mark.parametrize("which", ["dna", "qual"])
def test_bench_dna_qual_keys(ctx, bench_keys, which):
    dna, qual, off, pidx = bench_keys
    key0, idx = (dna, off) if which == "dna" else (qual, pidx)     # 4 zero pad bits, then the first 60 bits of the row
    _check(ctx, _rows_from_keys(key0, _tail(idx)))


def test_shared_top_bits(ctx):
    """The top 16 bits are the same for 99 % of the keys: that bucket is split again and again."""
    rng = np.random.default_rng(3)
    n = 2 * MSD_MIN_N + 4097
    key0 = (np.uint64(0xABCD) << np.uint64(48)) | rng.integers(0, 1 << 48, n, dtype=np.uint64)
    few = rng.random(n) < 0.01
    key0[few] = rng.integers(0, 1 << 63, few.sum(), dtype=np.uint64)
    _check(ctx, _rows_from_keys(key0, rng.integers(0, 4, size=(n, 4), dtype=np.uint8)))


def test_equal_keys(ctx):
    """All keys equal (no radix pass at all), then all but 0.1 % equal: that bucket outlives every digit and is cut into
    runs of equal keys."""
    rng = np.random.default_rng(4)
    n = MSD_MIN_N + 1
    tail = rng.integers(0, 3, size=(n, 5), dtype=np.uint8)
    key0 = np.full(n, 0x0123456789ABCDEF, dtype=np.uint64)
    _check(ctx, _rows_from_keys(key0, tail))
    few = rng.random(n) < 0.001
    key0[few] = rng.integers(0, 1 << 63, few.sum(), dtype=np.uint64)
    _check(ctx, _rows_from_keys(key0, tail))


def test_tiny_and_huge_buckets(ctx):
    rng = np.random.default_rng(5)
    n = 3 * MSD_MIN_N + 5
    key0 = rng.integers(0, 1 << 62, n, dtype=np.uint64)
    hot = rng.integers(0, 1 << 62, 3, dtype=np.uint64)
    for i, h in enumerate(hot):                           # three keys with 300 k, 100 k and 5 k copies, near neighbours too
        m = [300_000, 100_000, 5_000][i]
        at = rng.choice(n, m, replace=False)
        key0[at] = h ^ rng.integers(0, 4, m, dtype=np.uint64)
    _check(ctx, _rows_from_keys(key0, rng.integers(0, 256, size=(n, 8), dtype=np.uint8)))


@pytest.mark.parametrize("n", [MSD_MIN_N, MSD_MIN_N + 1, MSD_MIN_N + TILE - 1, MSD_MIN_N + 3 * TILE + 1000])
def test_sizes_near_threshold(ctx, n):
    rng = np.random.default_rng(n)
    t = rng.integers(0, 256, size=(n, 12), dtype=np.uint8)
    t[: n // 8, :2] = 7                                   # one top-16-bit bucket of n / 8 rows
    _check(ctx, t)
