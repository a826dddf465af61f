"""uqb_sort_rows (sort.cu, on the radix sort of prims.cu) against a stable numpy sort at the sizes and shapes of the
benched encode: tables made by the packer, whose round 0 sorts the packer's key0 through the MSD bucket path; every
refinement width class with tie groups of up to 32 rows and of more; narrow rows; the keyed encode members; the windowed
key scatter and wide gathers.

Every case asserts from the launch timers which kernels ran, and the last test checks that the cases together reached
every refinement kernel, so a threshold that moves cannot silently drop a class from these tests.

The reference is oracle.uq_vec.sort_unique_rows (lexsort over big-endian words).  An unmarked test pins it to
uq_vec.sort_unique, the void-view argsort / unique of the reference program."""
import numpy as np
import pytest

from oracle.uq_vec import sort_unique, sort_unique_rows
from test_symbol_paths import TILE_REC_MAX, assert_kernels, make_fastq

gpu = pytest.mark.gpu

MSD_MIN_N = 1 << 20
MSD = ("k_radix_hist_seg", "k_msd_plan", "k_bucket_sort")
SEEN = {}                 # kernel name -> launches, summed over the GPU cases of this module


def first_pass_kernel(width):
    """packed finisher right after round 0 (rows of 9..136 bytes without leading-zero offsets)"""
    if 9 <= width <= 40:
        return "k_small_groups_packed_8"
    if 41 <= width <= 72:
        return "k_small_groups_packed_16"
    if 73 <= width <= 136:
        return "k_small_groups_packed_32"
    return None


def rounds_kernel(width):
    """finisher of the refinement rounds"""
    return ("k_small_groups_8" if width <= 40 else "k_small_groups_16" if width <= 72 else
            "k_small_groups_32" if width <= 136 else "k_small_groups_64" if width <= 256 else "k_small_groups_gmem")


def lcp_kernel(width):
    return "k_group_lcp_8" if width <= 40 else "k_group_lcp_32"


# ------------------------------------------------------------------------------------------------
# reference and input builders (CPU)
# ------------------------------------------------------------------------------------------------
def _assert_same_as_void_sort(t):
    perm, key, ks, uniq = sort_unique_rows(t)
    perm_v, key_v, uniq_v = sort_unique(t)
    assert np.array_equal(perm, perm_v)
    assert np.array_equal(key, key_v)
    assert np.array_equal(ks, key_v[perm_v])
    assert np.array_equal(uniq, uniq_v)


@pytest.mark.parametrize("width", list(range(1, 18)) + [63, 64, 65, 255, 256, 257, 258])
def test_sort_unique_rows_equals_void_sort(width):
    rng = np.random.default_rng(width)
    n = 3_001
    t = rng.integers(0, 3, size=(n, width), dtype=np.uint8)
    t[rng.integers(0, n, n // 2)] = t[rng.integers(0, n, n // 2)]          # exact duplicates
    t[: n // 3, : max(width - 1, 1)] = t[0, : max(width - 1, 1)]           # rows that differ in their last byte only
    t[n // 3: n // 3 + 100, : width // 2] = 0                               # leading zero bytes
    t[-50:] = rng.integers(0, 256, size=(50, width), dtype=np.uint8)
    _assert_same_as_void_sort(t)


@pytest.mark.parametrize("width", [1, 7, 8, 9, 64, 257])
def test_sort_unique_rows_on_duplicates(width):
    rng = np.random.default_rng(100 + width)
    one = rng.integers(0, 256, size=(1, width), dtype=np.uint8)
    _assert_same_as_void_sort(np.repeat(one, 2_000, axis=0))              # one row, 2 000 times
    two = rng.integers(0, 256, size=(2, width), dtype=np.uint8)
    _assert_same_as_void_sort(two[rng.integers(0, 2, 2_000)])             # two rows, interleaved
    _assert_same_as_void_sort(one)                                        # a single row
    perm, key, ks, uniq = sort_unique_rows(np.zeros((0, width), np.uint8))
    assert len(perm) == len(key) == len(ks) == len(uniq) == 0 and uniq.shape == (0, width)


def tied_rows(n, width, seed, zeros=False):
    """n rows of `width` bytes in shuffled order:
      * tie groups, seven in ten of 2..32 rows, the others of 33..5 000 rows; the members of a group are one base row up
        to a chosen byte (the last byte for a third of the groups) and one of 1..64 variants from there on, so a group
        holds identical members and members that differ from that byte on;
      * one fifth staircase rows: a base row with one byte changed, the position running over the row;
      * zeros (rows wider than 256 bytes): two in three groups and the staircase start with a run of zero bytes, and a
        tenth of the rows are short right-aligned rows, as variable-length reads are packed."""
    rng = np.random.default_rng(seed)
    lo = 1 if zeros else 0                            # with zeros, the zero runs are the only zero bytes of the long rows
    n_stair, n_short = n // 5, (n // 10 if zeros else 0)
    n_grp = n - n_stair - n_short
    sizes, tot = [], 0
    while tot < n_grp:
        s = int(rng.integers(2, 33)) if rng.random() < 0.7 else int(rng.integers(33, 5_001))
        s = min(s, n_grp - tot)
        sizes.append(s)
        tot += s
    G = len(sizes)
    gid = np.repeat(np.arange(G), sizes)
    z = np.where(rng.random(G) < 2 / 3, rng.integers(0, width - 48, size=G), 0) if zeros else np.zeros(G, dtype=np.int64)
    cut = np.where(rng.random(G) < 1 / 3, width - 1, rng.integers(z + 8, width))
    nvar = rng.choice([1, 2, 3, 8, 64], size=G)
    voff = np.cumsum(nvar) - nvar
    base = rng.integers(lo, lo + 4, size=(G, width), dtype=np.uint8)
    var = rng.integers(lo, lo + 4, size=(int(nvar.sum()), width), dtype=np.uint8)
    vrow = voff[gid] + rng.integers(0, 1 << 30, size=n_grp) % nvar[gid]
    out = np.empty((n, width), dtype=np.uint8)
    pos = np.arange(width)
    for s0 in range(0, n_grp, 1 << 17):
        g = gid[s0:s0 + (1 << 17)]
        r = np.where(pos >= cut[g][:, None], var[vrow[s0:s0 + len(g)]], base[g])
        r[pos < z[g][:, None]] = 0
        out[s0:s0 + len(g)] = r
    zs = width // 2 if zeros else 0
    stair = np.repeat(rng.integers(lo, lo + 4, size=(1, width), dtype=np.uint8), n_stair, axis=0)
    stair[:, :zs] = 0
    i = np.arange(n_stair)
    stair[i, zs + 8 + i % (width - zs - 8)] = lo + 4 + i % 5
    out[n_grp:n_grp + n_stair] = stair
    if n_short:
        short = np.zeros((n_short, width), dtype=np.uint8)
        short[:, -40:] = rng.integers(1, 3, size=(n_short, 40), dtype=np.uint8)
        short[pos[None, :] < (width - rng.integers(1, 41, size=n_short))[:, None]] = 0
        out[n_grp + n_stair:] = short
    return out[rng.permutation(n)]


def pooled_fastq(n, pool, seed):
    """n records of 100 bp drawn by index from `pool` distinct make_fastq records (ACGT, ten quality symbols: rows of 25
    and 50 bytes); low indices are drawn thousands of times, high ones a few times.  The last quality symbol of a tenth
    of the records is redrawn, so copies of one record tie up to the last byte of their QUAL row."""
    recs = np.frombuffer(make_fastq(pool, 100, seed=seed), dtype=np.uint8).reshape(pool, -1)
    rng = np.random.default_rng(seed)
    out = recs[(pool * rng.random(n) ** 3).astype(np.int64)]
    sel = np.flatnonzero(rng.random(n) < 0.1)
    out[sel, -2] = np.frombuffer(b"ABCDEFGHIJ", dtype=np.uint8)[rng.integers(0, 10, len(sel))]    # before the last '\n'
    return out.tobytes()


def test_tied_rows_shapes():
    for width, zeros in ((40, False), (137, False), (264, True)):
        t = tied_rows(20_000, width, 1, zeros)
        assert t.shape == (20_000, width)
        _, key, _, uniq = sort_unique_rows(t)
        counts = np.bincount(key)
        assert counts.max() > 32 and (counts == 2).any() and len(uniq) < 20_000
        last = t[:, :-1].copy().view("V%d" % (width - 1)).reshape(-1)
        _, k1 = np.unique(last, return_inverse=True)
        assert len(np.unique(k1.reshape(-1))) < len(uniq)             # some rows tie up to their last byte
        if zeros:
            lead = np.argmax(t != 0, axis=1)
            assert lead.max() > 200 and (lead == 0).any()
        else:
            assert (t[:, 0] != 0).any()


def test_pooled_fastq_shape():
    from test_symbol_paths import np_pass1
    from uq_b200 import host
    data = pooled_fastq(5_000, 500, 3)
    assert len(data) // 5_000 <= TILE_REC_MAX
    dec = host.decide_alphabets(np_pass1(data))
    assert (dec["dna_bytes"], dec["qual_bytes"]) == (25, 50) and not dec["variable_read_lengths"]


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


@pytest.fixture(scope="module")
def refs():
    """(case, table) -> sort_unique_rows of the packed table: each reference is built once"""
    return {}


def _report(ctx):
    rep = ctx.timing_report()
    for k, v in rep.items():
        SEEN[k] = SEEN.get(k, 0) + v[0]
    return rep


def _need(ctx, gb):
    used, free, total = ctx.mem_info()
    if total - used < gb << 30:
        pytest.skip("needs ~%d GB of free HBM" % gb)


def _equal(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, "%s: shape %s, numpy %s" % (what, got.shape, want.shape)
    bad = np.flatnonzero((got != want).reshape(len(got), -1).any(axis=1)) if len(got) else []
    assert len(bad) == 0, "%s: %d of %d entries differ, first at %d (got %s, numpy %s)" % (
        what, len(bad), len(got), bad[0], got[bad[0]], want[bad[0]])


def check_sort(ctx, table, want, what, ran=(), absent=()):
    """sort_rows with all four outputs against want = sort_unique_rows of the table; the launch report must show `ran`
    and not `absent`"""
    perm_w, key_w, ks_w, uniq_w = want
    ctx.timing_reset()
    perm, key, uniq, nu, ks = ctx.sort_rows(table, want_perm=True, want_key=True, want_uniq=True, want_key_sorted=True)
    rep = _report(ctx)
    try:
        assert nu == len(uniq_w), "%s: %d unique rows, numpy %d" % (what, nu, len(uniq_w))
        _equal(perm.download(dtype=np.uint32), perm_w.astype(np.uint32), what + " perm")
        _equal(key.download(dtype=np.uint32), key_w.astype(np.uint32), what + " key")
        _equal(ks.download(dtype=np.uint32), ks_w.astype(np.uint32), what + " key_sorted")
        _equal(uniq.download().reshape(nu, table.width), uniq_w, what + " unique rows")
    finally:
        for a in (perm, key, uniq, ks):
            a.free()
    assert_kernels(rep, ran, absent, what)


# ---- tables made by the packer ------------------------------------------------------------------
N_PACK = 2_000_003
# case -> (read length, genome positions, quality pool, --pad) of the genome synth; "pooled": pooled_fastq
PACKED = {
    "bench": (150, N_PACK // 10, N_PACK // 5, False),         # the bench's duplication
    "deep": (150, N_PACK // 200, N_PACK // 200, False),       # most groups far longer than 32 rows
    "deep_pad": (150, N_PACK // 200, N_PACK // 200, True),    # QUAL of 150 bytes: no packed first pass
    "short": (32, N_PACK // 10, N_PACK // 5, False),          # DNA rows of exactly 8 bytes
    "long": (250, N_PACK // 200, N_PACK // 200, False),       # records too long for k_pack_tiles: no key0
    "pooled": None,                                            # QUAL rows of 50 bytes
}
WIDTHS = {"bench": (38, 113), "deep": (38, 113), "deep_pad": (38, 150), "short": (8, 24), "long": (63, 188),
          "pooled": (25, 50)}


def prepare_case(ctx, case):
    """host.prepare of the case's FASTQ -> (prepare's dict, what to free), with the packer asserted: k_pack_tiles (and
    so a key0 for every table of 8+ byte rows) where the records fit its tiles, k_pack_long for the 250 bp reads"""
    from uq_b200 import host
    if case == "pooled":
        data = pooled_fastq(N_PACK, 200_000, 5)
        fq, keep = ctx.load_fastq(data), []
    else:
        L, genome, pool, pad = PACKED[case]
        dev = ctx.synth("genome", N_PACK, L, 1002, genome=genome, pool=pool)
        fq, keep = ctx.adopt_fastq(dev), [dev]
    ctx.timing_reset()
    p = host.prepare(ctx, fq, pad=case == "deep_pad")
    rep = _report(ctx)
    assert (p["dna"].width, p["qual"].width) == WIDTHS[case]
    assert p["total"] == N_PACK
    if case == "long":
        assert fq.nbytes // N_PACK > TILE_REC_MAX
        assert_kernels(rep, ["k_pack_long"], ["k_pack_tiles"], "pack " + case)
    else:
        assert fq.nbytes // N_PACK <= TILE_REC_MAX
        assert_kernels(rep, ["k_pack_tiles"], ["k_pack_long", "k_pack_rows"], "pack " + case)
    return p, [p["dna"], p["qual"]] + p["cols"] + [fq] + keep


def _ref(refs, case, name, t):
    if (case, name) not in refs:
        refs[(case, name)] = sort_unique_rows(t)
    return refs[(case, name)]


@gpu
@pytest.mark.parametrize("name", ["dna", "qual"])
@pytest.mark.parametrize("case", list(PACKED))
def test_packer_tables(ctx, refs, case, name):
    """round 0 on the packer's key0 at n >= 2^20 (MSD buckets, k_chunk0_keys never runs), then the refinement: every
    output equals numpy's stable sort / unique of the downloaded table"""
    _need(ctx, 8)
    p, tmp = prepare_case(ctx, case)
    try:
        table = p[name]
        t = table.download()
        want = _ref(refs, case, name, t)
        w = table.width
        ran, absent = list(MSD), ["k_first_of_group"] if w <= 8 else ["k_uniq_from_keys"]
        if case == "long":
            ran.append("k_chunk0_keys")                       # no key0: k_pack_long does not write one
        else:
            absent.append("k_chunk0_keys")
        if w <= 8:
            ran.append("k_uniq_from_keys")                    # the unique rows are cut from the sorted keys
        elif first_pass_kernel(w):
            ran.append(first_pass_kernel(w))
        else:
            ran.append(rounds_kernel(w))
            absent += ["k_small_groups_packed_8", "k_small_groups_packed_16", "k_small_groups_packed_32"]
        if case in ("deep", "deep_pad", "long") and w > 8:    # tie groups of more than 32 rows that differ after byte 8
            ran += [rounds_kernel(w), lcp_kernel(w), "k_compact_active"]
        check_sort(ctx, table, want, "%s %s" % (case, name), ran, absent)
    finally:
        for a in tmp:
            a.free()


@gpu
@pytest.mark.parametrize("sort,raw", [("DNA", ()), ("QUAL", ()), ("DNA", ("QUAL", "QNAME")), ("QUAL", ("DNA",))])
def test_keyed_members_at_bench_path(ctx, refs, sort, raw):
    """run_mix on the deeply duplicated packer tables: every DNA / QUAL member and every QNAME_i.raw equals
    mix_dna_qual / mix_qname (uq_literal) computed through sort_unique_rows"""
    from uq_b200 import host
    _need(ctx, 8)
    p, tmp = prepare_case(ctx, "deep")
    try:
        tables = {"DNA": p["dna"].download(), "QUAL": p["qual"].download()}
        ref = {t: _ref(refs, "deep", t.lower(), tables[t]) for t in tables}
        cols = [c.download(dtype=m["dtype"]).reshape(-1) for c, m in zip(p["cols"], p["columns"])]
        s, r, pat = host.normalise_options(sort, list(raw) or None, None)
        ctx.timing_reset()
        members = host.run_mix(ctx, p["dna"], p["qual"], p["cols"], p["columns"], s, r, pat)
        rep = _report(ctx)
        got = members.download()
        members.free()
    finally:
        for a in tmp:
            a.free()
    order = ref[sort][0]
    for t in ("DNA", "QUAL"):
        _, key, _, uniq = ref[t]
        if t in raw:
            _equal(got[t + ".raw"], tables[t][order], "sort=%s %s.raw" % (sort, t))
        else:
            _equal(got[t], uniq, "sort=%s %s" % (sort, t))
            assert got[t + ".key"].dtype == np.min_scalar_type(len(uniq) - 1)
            _equal(got[t + ".key"].astype(np.int64), key[order], "sort=%s %s.key" % (sort, t))
    if "QNAME" in raw:
        for c, m in zip(cols, p["columns"]):
            assert got[m["name"] + ".raw"].dtype == np.dtype(m["dtype"])
            _equal(got[m["name"] + ".raw"], c[order], "sort=%s %s.raw" % (sort, m["name"]))
    assert_kernels(rep, MSD, [], "run_mix sort=%s raw=%s" % (sort, raw))


# ---- every width class on uploaded tables -------------------------------------------------------
@gpu
@pytest.mark.parametrize("n", [200_000, 1_200_007])
@pytest.mark.parametrize("width", [40, 41, 72, 73, 136, 137, 256, 257, 264])
def test_width_classes(ctx, width, n):
    """tie groups of 2..32 and of 33..5 000 rows and staircase rows in each width class of the refinement kernels, at a
    size below the MSD threshold and one above it (rows wider than 256 bytes: leading zero bytes, aux keys, LSD)"""
    _need(ctx, 4)
    t = tied_rows(n, width, seed=width * 7 + n % 97, zeros=width > 256)
    want = sort_unique_rows(t)
    packed = ["k_small_groups_packed_8", "k_small_groups_packed_16", "k_small_groups_packed_32"]
    ran = [rounds_kernel(width), lcp_kernel(width), "k_compact_active"]
    if width > 256:
        ran += ["k_leading_zero_bytes", "k_chunk0_keys_z"]
        absent = packed + ["k_chunk0_keys"]
    else:
        ran += ["k_chunk0_keys"] + ([first_pass_kernel(width)] if first_pass_kernel(width) else [])
        absent = [k for k in packed if k != first_pass_kernel(width)] + ["k_leading_zero_bytes"]
        if n >= MSD_MIN_N:
            ran += list(MSD)
    d = ctx.upload(t)
    try:
        check_sort(ctx, d, want, "width %d, %d rows" % (width, n), ran, absent)
    finally:
        d.free()


# ---- narrow rows at MSD size --------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("width", [1, 2, 3, 5, 7])
def test_narrow_rows(ctx, width):
    """1.5 M rows of 1..7 bytes, a few thousand distinct values: round-0 keys of `width` bytes, the unique rows cut from
    the sorted keys (k_uniq_from_keys writes `width` bytes per row).  Keys of 1 or 2 bytes have too few digits for the
    MSD path and take the LSD passes."""
    _need(ctx, 2)
    rng = np.random.default_rng(width)
    n = 1_500_001
    pool = rng.integers(0, 256, size=(min(5_000, 256 ** width), width), dtype=np.uint8)
    pool[0] = 0
    pool[-1] = 255
    t = pool[(len(pool) * rng.random(n) ** 2).astype(np.int64)]
    want = sort_unique_rows(t)
    ran = ["k_chunk0_keys", "k_uniq_from_keys"] + (list(MSD) if width >= 3 else [])
    d = ctx.upload(t)
    try:
        check_sort(ctx, d, want, "width %d" % width, ran, ["k_first_of_group", "k_small_groups_packed_8"])
    finally:
        d.free()


# ---- windowed key scatter, gathers, wide unique rows --------------------------------------------
@gpu
def test_key_scatter_in_windows(ctx):
    """want_key above 3 * 2^23 rows: the key goes out through the window-regrouped scatter (k_pairs_apply)"""
    _need(ctx, 4)
    rng = np.random.default_rng(11)
    n = 3 * (1 << 23) + 12_345
    pool = rng.integers(0, 256, size=(1_000_000, 5), dtype=np.uint8)
    t = pool[rng.integers(0, len(pool), n)]
    _, key_w, _, uniq_w = sort_unique_rows(t)
    d = ctx.upload(t)
    ctx.timing_reset()
    _, key, _, nu = ctx.sort_rows(d, want_key=True)
    rep = _report(ctx)
    try:
        assert nu == len(uniq_w)
        _equal(key.download(dtype=np.uint32), key_w.astype(np.uint32), "key")
    finally:
        key.free()
        d.free()
    assert_kernels(rep, ["k_pairs_apply"] + list(MSD), ["k_scatter_key"], "key scatter")


GATHER_KERNEL = {1: "k_gather_items<uint8_t>", 2: "k_gather_items<uint16_t>", 4: "k_gather_items<uint32_t>",
                 8: "k_gather_items<uint64_t>"}


@gpu
@pytest.mark.parametrize("width", [1, 2, 3, 4, 8, 15, 16, 17, 127, 128, 129, 1024, 1025, 4097])
def test_gather_rows(ctx, width):
    rng = np.random.default_rng(width)
    m, n = (5_003, 20_011) if width > 1024 else (50_001, 100_003)
    t = rng.integers(0, 256, size=(m, width), dtype=np.uint8)
    idx = rng.integers(0, m, n).astype(np.uint32)
    idx[:3] = [m - 1, 0, m - 1]
    d, di = ctx.upload(t), ctx.upload(idx)
    ctx.timing_reset()
    out = ctx.gather_rows(d, di)
    rep = _report(ctx)
    try:
        _equal(out.download().reshape(n, width), t[idx], "gather width %d" % width)
    finally:
        for a in (d, di, out):
            a.free()
    kernel = GATHER_KERNEL.get(width) or ("k_gather_narrow" if width <= 16 else "k_gather_rows32" if width <= 1024
                                          else "k_gather_rows")
    assert_kernels(rep, [kernel], [], "gather width %d" % width)


@gpu
def test_wide_unique_rows(ctx):
    """300 k right-aligned rows of 2 000 bytes, 60 k distinct: unique rows gathered one warp per row (k_gather_rows)"""
    _need(ctx, 4)
    rng = np.random.default_rng(12)
    n, width = 300_007, 2_000
    pool = rng.integers(1, 4, size=(60_000, width), dtype=np.uint8)
    pool[np.arange(width)[None, :] < (width - rng.integers(1, width + 1, size=60_000))[:, None]] = 0
    pool[:100, :-1] = pool[0, :-1]                                # rows that differ in the last byte only
    t = pool[(len(pool) * rng.random(n) ** 2).astype(np.int64)]
    want = sort_unique_rows(t)
    d = ctx.upload(t)
    try:
        check_sort(ctx, d, want, "width 2000", ["k_leading_zero_bytes", "k_first_of_group", "k_gather_rows"],
                   ["k_uniq_from_keys"])
    finally:
        d.free()


# ---- coverage guard -----------------------------------------------------------------------------
REQUIRED = ("k_small_groups_packed_8", "k_small_groups_packed_16", "k_small_groups_packed_32",
            "k_small_groups_8", "k_small_groups_16", "k_small_groups_32", "k_small_groups_64", "k_small_groups_gmem",
            "k_group_lcp_8", "k_group_lcp_32", "k_leading_zero_bytes", "k_compact_active", "k_uniq_from_keys",
            "k_pairs_apply") + MSD


@gpu
def test_every_sort_path_ran(request):
    """the cases above, together, launched every refinement kernel, k_uniq_from_keys, k_pairs_apply and the MSD kernels
    (runs when the whole module is selected)"""
    mod = request.module
    cases = {name for name, f in vars(mod).items() if name.startswith("test_") and f is not test_every_sort_path_ran
             and any(m.name == "gpu" for m in getattr(f, "pytestmark", []))}
    selected = {getattr(i, "originalname", i.name) for i in request.session.items if getattr(i, "module", None) is mod}
    if not cases <= selected:
        pytest.skip("only a part of the module was selected")
    missing = [k for k in REQUIRED if not SEEN.get(k)]
    assert not missing, "no case of this module launched %s" % missing
