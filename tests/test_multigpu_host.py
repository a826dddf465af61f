"""Host-side merges of the multi-GPU global encode (uq_b200/multigpu.py) on CPU: per-shard statistics produced
by the contract emulation must merge into exactly the statistics of the whole file; the object collectives run
over 2 gloo ranks."""
import os
import socket

import numpy as np
import pytest

from conftest import golden_case, load_manifest
from emu import emu_colstats, emu_stats
from uq_b200 import _lib as L, host, multigpu as mg
from test_gpu_parity import STAT_FIELDS, STAT_SCALARS

CASES = ["c2_keyed_sortDNA", "c3_casava_sortQNAME", "c7_offset_suffix_keyed", "c6_checkpoints", "c5_variable_raw"]


def shards_of(fq, cuts):
    lines = fq.split(b"\n")[:-1]
    recs = [b"\n".join(lines[i:i + 4]) + b"\n" for i in range(0, len(lines), 4)]
    bounds = [0] + [int(len(recs) * c) for c in cuts] + [len(recs)]
    return [(b"".join(recs[a:b]), a, b - a) for a, b in zip(bounds[:-1], bounds[1:])]


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("cuts", [(0.5,), (0.6, 0.61, 0.9)])
def test_merged_statistics_equal_whole_file_statistics(name, cuts):
    fq, _, kw = golden_case(name)
    shards = shards_of(fq, cuts)
    ref = fq.split(b"\n")[0]
    parts = []
    for data, base, n in shards:
        st, _ = emu_stats(data, ref=ref, base=base)
        parts.append((mg.stats_to_plain(st), base, n))
    parts[0][0]["first_name"] = ref
    got = mg.merge_stats(parts)
    want, n_total = emu_stats(fq)
    for f in STAT_SCALARS:
        assert getattr(got, f) == getattr(want, f), f
    for f in STAT_FIELDS:
        assert list(getattr(got, f)) == list(getattr(want, f)), f
    prefix, suffix, seps = host.derive_qname_layout(got, n_total)
    # column statistics and dictionaries
    whole_cols, bad, whole_dicts = emu_colstats(fq, len(prefix), len(suffix), seps)
    ncols = len(seps) + 1
    early = [whole_cols[c].n_distinct == L.U64_MAX for c in range(ncols)]
    plains, dicts = [], []
    for data, base, n in shards:
        cols, bad, _ = emu_colstats(data, len(prefix), len(suffix), seps)
        plains.append(mg.colstats_to_plain(cols, ncols))
        # local dictionaries with global first occurrences, computed directly
        toks = [l.split(b"\n")[0] for l in data.split(b"\n")[0::4][:-1]]
        d = {}
        for c in range(ncols):
            if early[c]:
                continue
            first = {}
            for r, name_line in enumerate(data.split(b"\n")[0::4][:n]):
                mid = name_line[len(prefix):len(name_line) - len(suffix)].decode("latin-1")
                import re
                tok = re.split("(.*)".join(seps), mid)[c]
                first.setdefault(tok, base + r)
            ks = sorted(first)
            d[c] = (ks, [first[k] for k in ks])
        dicts.append(d)
    if n_total > 10000 and shards[0][2] < 10001:
        pytest.skip("rank 0 would not hold checkpoint 0")
    # rank 0's checkpoint-0 value is the global one for early-demoted columns
    for c in range(ncols):
        if early[c]:
            plains[0][c]["distinct_at"][0] = int(whole_cols[c].distinct_at[0])
    merged, gd = mg.merge_colstats(plains, n_total, early, dicts)
    for c in range(ncols):
        for f in ("all_int", "all_canonical", "overflow", "min_len", "max_len", "n_distinct", "n_checkpoints"):
            assert getattr(merged[c], f) == getattr(whole_cols[c], f), (c, f)
        if whole_cols[c].all_int:
            assert (merged[c].min_val, merged[c].max_val) == (whole_cols[c].min_val, whole_cols[c].max_val)
        assert list(merged[c].distinct_at) == list(whole_cols[c].distinct_at), c
        if c in whole_dicts:
            assert gd[c] == whole_dicts[c]
    assert host.decide_columns(merged, n_total, lambda i: gd[i]) == host.decide_columns(whole_cols, n_total, lambda i: whole_dicts[i])


def test_pick_splitters_is_deterministic_and_sorted():
    rng = np.random.default_rng(3)
    s = rng.integers(0, 4, size=(500, 5), dtype=np.uint8)
    a = mg.pick_splitters(s, 4)
    b = mg.pick_splitters(s[rng.permutation(500)], 4)
    assert a.shape == (3, 5) and np.array_equal(a, b)
    v = a.view("V5").reshape(-1)
    assert np.array_equal(np.sort(v), v)
    assert mg.pick_splitters(np.zeros((0, 5), np.uint8), 4).shape == (0, 5)
    assert mg.n_checkpoints(10000) == 0 and mg.n_checkpoints(10001) == 1 and mg.n_checkpoints(20001) == 2


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    comm = mg.Comm(dist, "cpu")
    fq, _, _ = golden_case("c3_casava_sortQNAME")
    data, base, n = shards_of(fq, (0.4,))[rank]
    ref = comm.all_gather_object(data.split(b"\n")[0])[0]
    st, _ = emu_stats(data, ref=ref, base=base)
    parts = comm.all_gather_object((mg.stats_to_plain(st), base, n))
    parts[0][0]["first_name"] = ref
    merged = mg.merge_stats(parts)
    recv = comm.exchange_counts([10 * rank + k for k in range(world)])
    if rank == 0:
        q.put((host.derive_qname_layout(merged, 700), recv))
    dist.destroy_process_group()


def test_object_collectives_over_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs: p.start()
    layout, recv = q.get(timeout=120)
    for p in procs: p.join(timeout=60)
    assert all(p.exitcode == 0 for p in procs)
    assert layout == ("@EAS139:136:FC706VJ:", "", "::: :::")
    assert recv == [0, 10]          # rank 0 receives send_counts[0] of rank 0 (=0) and of rank 1 (=10)


def _board_worker(rank, world, port, q, use_board):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      UQB_MG_SHM="1" if use_board else "0")
    dist.init_process_group("gloo", rank=rank, world_size=world)
    comm = mg.Comm(dist, "cpu")
    ok = (comm.board is not None) == use_board
    for k in range(300):                                  # many rounds back to back: the two-slot protocol must never mix rounds
        got = comm.all_gather_object((rank, k, b"x" * ((k * 37 + rank) % 5000)))
        ok = ok and [g[:2] for g in got] == [(r, k) for r in range(world)] and all(len(g[2]) == (k * 37 + r) % 5000 for r, g in enumerate(got))
    big = np.arange(400_000 + rank, dtype=np.int64)       # 3.2 MB: does not fit a slot -> the round falls back to gloo
    got = comm.all_gather_object(big if rank == 1 else rank)
    ok = ok and got[0] == 0 and len(got[1]) == 400_001
    got = comm.all_gather_object({"after": rank})          # and the board is usable again afterwards
    ok = ok and got == [{"after": r} for r in range(world)]
    calls = comm.host_collectives[0]
    comm.close()
    q.put((rank, ok, calls))
    dist.destroy_process_group()


@pytest.mark.parametrize("use_board", [True, False])
def test_shared_memory_board_matches_gloo(use_board):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    world = 3
    procs = [ctx.Process(target=_board_worker, args=(r, world, port, q, use_board)) for r in range(world)]
    for p in procs: p.start()
    res = sorted(q.get(timeout=180) for _ in range(world))
    for p in procs: p.join(timeout=60)
    assert all(p.exitcode == 0 for p in procs)
    assert res == [(r, True, 302) for r in range(world)]


# ---- partition-first sample sort: the host side of global_unique, emulated with numpy ---------------------------
def _emu_partition(rows, split_keys):
    """contract of uqb_partition_positions: dest = number of splitter keys <= big-endian first 8 bytes; stable grouping
    (order = pos^-1)"""
    key = mg.row_key64(rows)
    dest = np.searchsorted(np.asarray(split_keys, dtype=np.uint64), key, side="right")
    order = np.argsort(dest, kind="stable")
    return order, np.bincount(dest, minlength=len(split_keys) + 1)


def test_row_key64_is_the_big_endian_prefix():
    rows = np.array([[1, 2, 3, 4, 5, 6, 7, 8, 9], [0, 0, 0, 0, 0, 0, 0, 1, 255], [255] * 9], dtype=np.uint8)
    assert mg.row_key64(rows).tolist() == [0x0102030405060708, 1, 0xFFFFFFFFFFFFFFFF]
    narrow = np.array([[1, 2, 3], [0, 0, 9]], dtype=np.uint8)                 # shorter than 8 bytes: zero padded on the right
    assert mg.row_key64(narrow).tolist() == [0x0102030000000000, 0x0000090000000000]
    assert mg.row_key64(np.zeros((0, 5), np.uint8)).shape == (0,)


@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("width", [3, 9, 38])
def test_partition_first_sample_sort_gives_the_global_sort(world, width):
    """rows scattered over `world` ranks, partitioned by the splitter keys and sorted per destination: the
    concatenation over the destinations is the stable global sort, identical rows meet on one rank, and the ids
    scattered back through the partition order are numpy.unique's inverse."""
    rng = np.random.default_rng(world * 100 + width)
    n = 4000
    table = rng.integers(0, 3, size=(n, width), dtype=np.uint8)              # few byte values: many ties on 8-byte prefixes
    table[rng.integers(0, n, 300)] = table[rng.integers(0, n, 300)]          # and exact duplicates
    cuts = np.sort(rng.integers(1, n - 1, world - 1))
    shards = np.split(np.arange(n), cuts)
    samples = [table[s][np.unique(np.linspace(0, len(s) - 1, num=min(len(s), 64)).astype(np.int64))] for s in shards]
    splitters = mg.pick_splitters(np.concatenate(samples), world)
    skeys = np.sort(mg.row_key64(splitters))
    received = [[] for _ in range(world)]                                     # (global record index, row) per destination
    routes = []
    for s in shards:
        order, counts = _emu_partition(table[s], skeys)
        routes.append((s, order, counts))
        b = np.concatenate([[0], np.cumsum(counts)])
        for d in range(world):
            for j in order[b[d]:b[d + 1]]:
                received[d].append((int(s[j]), table[s[j]]))
    void = lambda a: np.ascontiguousarray(a).view("V%d" % width).reshape(-1)
    want_perm = np.argsort(void(table), kind="stable")
    got_perm, uniq_parts, ids = [], [], np.zeros(n, dtype=np.int64)
    offset = 0
    for d in range(world):
        if not received[d]:
            continue
        idx = np.array([g for g, _ in received[d]])
        rows = np.stack([r for _, r in received[d]])
        p = np.argsort(void(rows), kind="stable")
        got_perm.extend(idx[p].tolist())
        u, inv = np.unique(void(rows), return_inverse=True)
        uniq_parts.append(u)
        ids[idx] = inv.reshape(-1) + offset
        offset += len(u)
    assert got_perm == want_perm.tolist()                                     # rank-major concatenation = stable global sort
    wu, winv = np.unique(void(table), return_inverse=True)
    assert np.array_equal(np.concatenate(uniq_parts), wu)                     # unique tables concatenate
    assert np.array_equal(ids, winv.reshape(-1))                              # ids back in record order


def test_skew_guard_constants():
    assert mg.SKEW_LIMIT >= 1.5 and mg.SAMPLES_PER_RANK >= 256
