"""One uQ container from N GPUs (SURVEY section 8e): every rank holds a contiguous range of the reads of ONE
FASTQ file and the result is bit-identical to the single-GPU encode of the whole file.

  phase                      what crosses ranks
  -------------------------  --------------------------------------------------------------------------
  split                      all-gather of the per-rank read counts (object collective)
  Pass-1 statistics          every rank measures against the GLOBAL first QNAME line (uqb_fastq_set_reference);
                             the O(alphabet) structs are all-gathered and merged on the host (merge_stats)
  QNAME column typing        all-gather + merge of the per-column statistics and of the dictionaries of the
                             columns that stay 'mapping' (merge_colstats)
  pack / column encode       nothing (per read)
  sort / unique              partition-first sample sort: splitters from gathered row samples, every row goes to
                             the rank whose range holds its first 8 bytes (ONE all-to-all of the rows, NCCL over
                             NVLink), the rank sorts / uniques its range once, the global ids return through the
                             reverse all-to-all (global_unique; global_unique_merge is the skew-proof variant)
  --sort order               the per-record payload (keys / raw rows) follows the rows of the sorted-on table:
                             same partition, same all-to-all, then the receiver's stable argsort (global_order)

The device collectives go through torch.distributed (NCCL) on zero-copy tensor views of the arena memory
(`__cuda_array_interface__`); the host-side merges are plain Python over tiny structs and are covered by
2-rank gloo tests on CPU.
"""
import os

import numpy as np

from . import _lib as L
from . import host

_ARRAY_FIELDS = ("base_count", "qual_count", "base_single_qual", "last_count_mismatch", "first_lcp_eq", "first_lcs_eq",
                 "first_short_prefix", "first_short_suffix")
_SCALAR_FIELDS = ("dna_min", "dna_max", "bad_first_char", "bad_plus_record", "bad_len_record", "first_len", "last_len",
                  "max_name_len", "prefix_len", "suffix_len")


# ------------------------------------------------------------------------------------------------
# host-side merges (no device, no torch)
# ------------------------------------------------------------------------------------------------
def stats_to_plain(st):
    d = {f: list(getattr(st, f)) for f in _ARRAY_FIELDS}
    d.update({f: int(getattr(st, f)) for f in _SCALAR_FIELDS})
    d["first_name"] = bytes(st.first_name[:st.first_len])
    d["last_name"] = bytes(st.last_name[:st.last_len])
    return d


def merge_stats(parts):
    """parts: [(plain stats measured against the global line 1, first global record, number of records)] in rank
    order, empty shards skipped by the caller -> uqb_stats of the whole file."""
    st = L.Stats()
    ref_len = len(parts[0][0]["first_name"])
    for i in range(256):
        st.base_single_qual[i] = -1
        st.last_count_mismatch[i] = -1
    for j in range(L.HDR_MAX + 1):
        st.first_lcp_eq[j] = st.first_lcs_eq[j] = st.first_short_prefix[j] = st.first_short_suffix[j] = L.NONE_I64
    st.bad_plus_record = st.bad_len_record = -1
    dmin, dmax, mname = None, 0, 0
    for p, base, n in parts:
        for i in range(256):
            st.base_count[i] += p["base_count"][i]
            st.qual_count[i] += p["qual_count"][i]
            a, b = st.base_single_qual[i], p["base_single_qual"][i]
            st.base_single_qual[i] = b if a == -1 else (a if b == -1 or b == a else 256)
            if p["last_count_mismatch"][i] >= 0:
                st.last_count_mismatch[i] = max(st.last_count_mismatch[i], base + p["last_count_mismatch"][i])
        for f in ("first_lcp_eq", "first_lcs_eq", "first_short_prefix", "first_short_suffix"):
            dst = getattr(st, f)
            for j in range(ref_len + 1):
                v = p[f][j]
                if v != L.NONE_I64:
                    dst[j] = min(dst[j], base + v)
        for f in ("bad_plus_record", "bad_len_record"):
            v = p[f]
            if v >= 0:
                cur = getattr(st, f)
                setattr(st, f, base + v if cur < 0 else min(cur, base + v))
        dmin = p["dna_min"] if dmin is None else min(dmin, p["dna_min"])
        dmax = max(dmax, p["dna_max"])
        mname = max(mname, p["max_name_len"])
    first, last = parts[0][0]["first_name"], parts[-1][0]["last_name"]
    st.first_len, st.last_len = len(first), len(last)
    for i, b in enumerate(first): st.first_name[i] = b
    for i, b in enumerate(last): st.last_name[i] = b
    st.bad_first_char = parts[0][0]["bad_first_char"]
    st.dna_min, st.dna_max, st.max_name_len = dmin, dmax, mname
    pl = sl = ref_len
    for j in range(ref_len + 1):
        if st.first_lcp_eq[j] != L.NONE_I64: pl = min(pl, j)
        if st.first_lcs_eq[j] != L.NONE_I64: sl = min(sl, j)
    st.prefix_len, st.suffix_len = pl, sl
    return st


def colstats_to_plain(cols, ncols):
    out = []
    for c in range(ncols):
        cs = cols[c]
        out.append(dict(all_int=int(cs.all_int), all_canonical=int(cs.all_canonical), overflow=int(cs.overflow),
                        min_val=int(cs.min_val), max_val=int(cs.max_val), min_len=int(cs.min_len), max_len=int(cs.max_len),
                        n_distinct=int(cs.n_distinct), distinct_at=list(cs.distinct_at)))
    return out


def n_checkpoints(n_total):
    k, t = 0, 10000
    while t <= n_total - 1 and k < L.MAX_CHECKPOINTS:
        k += 1
        t *= 2
    return k


def merge_colstats(parts, n_total, early_demoted, dictionaries):
    """parts: per rank [plain colstats per column]; early_demoted[c]: the column left 'mapping' at checkpoint 0
    (decided on the rank that holds records 0..10000); dictionaries: per rank {column: (tokens, first global
    record of each token)} for the other columns -> (uqb_colstats array of the whole file, {column: sorted
    global dictionary})."""
    ncols = len(parts[0])
    cols = (L.ColStats * ncols)()
    ncheck = n_checkpoints(n_total)
    merged_dicts = {}
    for c in range(ncols):
        cs = cols[c]
        ps = [p[c] for p in parts]
        cs.all_int = int(all(p["all_int"] for p in ps))
        cs.all_canonical = int(all(p["all_canonical"] for p in ps))
        cs.overflow = int(any(p["overflow"] for p in ps))
        cs.min_val = min(p["min_val"] for p in ps)
        cs.max_val = max(p["max_val"] for p in ps)
        cs.min_len = min(p["min_len"] for p in ps)
        cs.max_len = max(p["max_len"] for p in ps)
        cs.n_checkpoints = ncheck
        if early_demoted[c]:
            cs.distinct_at[0] = parts[0][c]["distinct_at"][0]
            for k in range(1, L.MAX_CHECKPOINTS): cs.distinct_at[k] = L.U64_MAX
            cs.n_distinct = L.U64_MAX
            continue
        first = {}
        for d in dictionaries:
            toks, occ = d[c]
            for t, o in zip(toks, occ):
                o = int(o)
                if t not in first or o < first[t]:
                    first[t] = o
        t = 10000
        for k in range(ncheck):
            cs.distinct_at[k] = sum(1 for o in first.values() if o <= t)
            t *= 2
        cs.n_distinct = len(first)
        merged_dicts[c] = sorted(first)
    return cols, merged_dicts


def pick_splitters(all_samples, world):
    """all_samples: uint8 [m][w] (gathered, any order) -> the world-1 splitter rows (identical on every rank)."""
    m, w = all_samples.shape
    if m == 0 or world == 1:
        return np.zeros((0, w), dtype=np.uint8)
    v = np.ascontiguousarray(all_samples).view("V%d" % w).reshape(-1) if w else np.zeros(m, dtype="V1")
    order = np.argsort(v, kind="stable")
    pos = [min(m - 1, (k * m) // world) for k in range(1, world)]
    return np.ascontiguousarray(all_samples[order[pos]])


# ------------------------------------------------------------------------------------------------
# diagnostics: UQB_MG_TRACE=1 prints wall-clock milliseconds per phase on rank 0 (adds device syncs)
# ------------------------------------------------------------------------------------------------
import time as _time
_TRACE = {"on": os.environ.get("UQB_MG_TRACE") == "1", "t": 0.0, "log": []}


def _mark(ctx, comm, name):
    if not _TRACE["on"]:
        return
    ctx.sync()
    now = _time.perf_counter()
    if name is not None and comm.rank == 0:
        _TRACE["log"].append((name, round((now - _TRACE["t"]) * 1e3, 2)))
    _TRACE["t"] = _time.perf_counter()


def trace_dump():
    out, _TRACE["log"] = _TRACE["log"], []
    return out


# ------------------------------------------------------------------------------------------------
# communication
# ------------------------------------------------------------------------------------------------
def _segmented(ctx, table, router, seg_counts, align=128):
    """the rows of `table` grouped by destination in a byte buffer with aligned segments.  router = [pos] from
    uqb_partition_positions: rows of 1 .. Context.SCATTER_MAX_WIDTH bytes are scattered by pos (streaming), other widths
    are gathered through order = pos^-1, which is computed on first use and kept as router[1]."""
    pos = router[0]
    if 0 < table.width <= ctx.SCATTER_MAX_WIDTH:
        return ctx.scatter_rows_segmented(table, pos, seg_counts, align)
    if len(router) < 2:
        iota = ctx.upload(np.arange(pos.n, dtype=np.uint32))
        router.append(ctx.scatter_u32(iota, pos))
        iota.free()
    return ctx.gather_rows_segmented(table, router[1], seg_counts, align)


def _router_free(router):
    for a in router:
        a.free()


class PeerWindow:
    """Receive memory that every rank can write: ptrs[r] is the device address, valid in THIS process, of rank r's buffer
    (symmetric / peer-mapped memory over NVLink; for the emulated ranks of LocalComm plain pointers of the one device).
    The buffer is cut into `slots` equal slots which the row exchanges use round-robin - every rank runs the same
    sequence of exchanges, so the slot of an exchange needs no agreement.  barrier() is ordered on the context's stream
    and spans all ranks: before an exchange it says that nobody reads the slot's previous contents any more, after it
    that all rows have landed."""

    def __init__(self, ptrs, rank, nbytes, slots, barrier, keep=None):
        self.ptrs, self.rank, self.slots = [int(p) for p in ptrs], rank, slots
        self.slot_bytes = nbytes // slots // 256 * 256
        self.barrier = barrier
        self.seq = 0
        self._keep = keep

    def next_slot(self):
        base = (self.seq % self.slots) * self.slot_bytes
        self.seq += 1
        return base


def open_peer_window(dist, device, stream, nbytes, slots=3):
    """torch symmetric memory (CUDA VMM handles exchanged through the process group's store): one allocation per rank,
    mapped into every other rank of the node.  Collective; call it once, outside the timed loop."""
    import torch
    import torch.distributed._symmetric_memory as symm_mem
    buf = symm_mem.empty(int(nbytes), dtype=torch.uint8, device=device)
    hdl = symm_mem.rendezvous(buf, dist.group.WORLD)

    def barrier():
        if stream is not None:
            with torch.cuda.stream(stream):
                hdl.barrier(channel=0)
        else:
            hdl.barrier(channel=0)
            torch.cuda.current_stream().synchronize()
    return PeerWindow(list(hdl.buffer_ptrs), dist.get_rank(), int(nbytes), slots, barrier, keep=(buf, hdl))


def _p2p_plan(comm, ctx, table, router, count_table):
    """-> (slot base, destination address of this rank's rows in every rank's slot) when the exchange can go through the
    peer window, else None.  Decided from the count table alone, so every rank decides alike."""
    win = getattr(comm, "window", None)
    w = table.width
    if win is None or count_table is None or not (0 < w <= ctx.SCATTER_MAX_WIDTH):
        return None
    world = comm.world
    if max(sum(count_table[s][d] for s in range(world)) for d in range(world)) * w > win.slot_bytes:
        return None
    base = win.next_slot()
    return base, [win.ptrs[d] + base + sum(count_table[s][d] for s in range(comm.rank)) * w for d in range(world)]


def _p2p_exchange(comm, ctx, table, router, send_counts, recv_counts, plan):
    base, addrs = plan
    recv = ctx.wrap(comm.window.ptrs[comm.rank] + base, sum(recv_counts), table.width)
    comm.window.barrier()                                # nobody reads what the slot held before
    ctx.scatter_rows_to(table, router[0], send_counts, addrs)
    return dict(p2p=True, recv=recv)


class ShmBoard:
    """all_gather of small python objects between the ranks of ONE node through a POSIX shared-memory segment: every rank
    owns two slots (round parity) and a header (sequence number, size); a round is: pickle into my slot, publish the
    sequence number, spin until every rank has published it, unpickle theirs.  A rank can run at most one round ahead of
    the slowest reader (it needs that reader's next header to finish its own next round), so two slots are enough.
    Latency is tens of microseconds where gloo's all_gather_object (two TCP collectives + pickling on both sides) takes
    0.3-2 ms; encode_sharded issues about a dozen of them per step, each one with an idle GPU behind it.  An object that
    does not fit its slot is flagged in the header and the round is repeated over the fallback collective."""
    SLOT = 1 << 20
    HDR = 64

    def __init__(self, name, rank, world, create):
        from multiprocessing import shared_memory
        size = world * (self.HDR + 2 * self.SLOT)
        self.shm = shared_memory.SharedMemory(name=name, create=create, size=size)
        if not create:
            # the creator unlinks; keep the resource tracker of the other ranks from doing it a second time
            try:
                from multiprocessing import resource_tracker
                resource_tracker.unregister(self.shm._name, "shared_memory")
            except Exception:
                pass
        self.rank, self.world, self.seq, self.owner = rank, world, 0, create
        self.hdr = np.ndarray((world, self.HDR // 8), dtype=np.int64, buffer=self.shm.buf, offset=0)
        self.data0 = world * self.HDR
        if create:
            self.hdr[:] = 0

    def _slot(self, r, parity):
        o = self.data0 + (2 * r + parity) * self.SLOT
        return self.shm.buf[o:o + self.SLOT]

    def all_gather(self, obj, fallback):
        import pickle
        self.seq += 1
        seq, par = self.seq, self.seq & 1
        blob = pickle.dumps(obj, protocol=pickle.HIGHEST_PROTOCOL)
        big = len(blob) > self.SLOT
        if not big:
            self._slot(self.rank, par)[:len(blob)] = blob
        self.hdr[self.rank, 1 + par] = -1 if big else len(blob)
        self.hdr[self.rank, 0] = seq                                     # publish (x86: stores stay in order)
        out, any_big = [None] * self.world, big
        deadline = _time.monotonic() + 600.0
        for r in range(self.world):
            spins = 0
            while self.hdr[r, 0] < seq:
                spins += 1
                if spins > 2000:
                    _time.sleep(0.00005)
                    if _time.monotonic() > deadline:
                        raise RuntimeError("ShmBoard: rank %d did not reach round %d" % (r, seq))
            nb = int(self.hdr[r, 1 + par])
            if nb < 0:
                any_big = True
            elif not any_big:
                out[r] = pickle.loads(bytes(self._slot(r, par)[:nb]))
        return fallback(obj) if any_big else out

    def close(self):
        try:
            self.hdr = None
            self.shm.close()
            if self.owner:
                self.shm.unlink()
        except Exception:
            pass


class Comm:
    """torch.distributed behind four calls; `dist=None` is the single-rank case."""

    def __init__(self, dist=None, device=None, stream=None):
        """stream: the torch.cuda.Stream whose cuda_stream the Context was created on.  With it the exchanges are ordered
        on the device (the collective waits for the rows on that stream, the stream waits for the collective) and the host
        never blocks around them; without it every exchange is bracketed by host synchronisations."""
        self.dist, self.device, self.stream = dist, device, stream
        self.window = None                               # PeerWindow: row exchanges as direct stores into the peers' memory
        self.rank = dist.get_rank() if dist else 0
        self.world = dist.get_world_size() if dist else 1
        # the small object collectives run over gloo next to NCCL: queued on the NCCL communicator they would wait
        # behind a row exchange that is still in flight and serialise the pipeline of encode_sharded
        self.obj_group = None
        if dist and dist.get_backend() == "nccl":
            self.obj_group = dist.new_group(backend="gloo")
        self.board = None                                # ShmBoard when all ranks share this node
        self.host_collectives = [0, 0.0]                 # calls, seconds spent inside them (latency + waiting for the slowest rank)
        if dist and self.world > 1 and os.environ.get("UQB_MG_SHM", "1") != "0":
            self._open_board()

    def _open_board(self):
        import socket, uuid
        name = "uqb_%s" % uuid.uuid4().hex[:16] if self.rank == 0 else None
        info = self._gloo_gather((socket.gethostname(), name))
        if len({h for h, _ in info}) != 1:               # several nodes: gloo stays
            return
        name = info[0][1]
        try:
            if self.rank == 0:
                self.board = ShmBoard(name, 0, self.world, create=True)
            self.dist.barrier(group=self.obj_group)
            if self.rank != 0:
                self.board = ShmBoard(name, self.rank, self.world, create=False)
            ok = self.board is not None
        except Exception:
            ok = False
        if not all(self._gloo_gather(ok)):
            if self.board:
                self.board.close()
            self.board = None

    def _gloo_gather(self, obj):
        out = [None] * self.world
        self.dist.all_gather_object(out, obj, group=self.obj_group)
        return out

    def all_gather_object(self, obj):
        if not self.dist:
            return [obj]
        t0 = _time.perf_counter()
        out = self.board.all_gather(obj, self._gloo_gather) if self.board is not None else self._gloo_gather(obj)
        self.host_collectives[0] += 1
        self.host_collectives[1] += _time.perf_counter() - t0
        return out

    def close(self):
        if self.board is not None:
            self.board.close()
            self.board = None

    def exchange_counts(self, send_counts):
        """send_counts[k] = rows this rank sends to rank k -> rows it receives from every rank"""
        table = self.all_gather_object(list(map(int, send_counts)))
        return [table[src][self.rank] for src in range(self.world)]

    def _tensor(self, arr):
        import torch
        if arr.nbytes == 0:
            return torch.empty(0, dtype=torch.uint8, device=self.device)
        return torch.as_tensor(arr, device=self.device)

    def _issue(self, ctx, fn):
        """run a torch.distributed call after the work queued on the context's stream"""
        import torch
        if self.stream is None or _TRACE["on"]:
            ctx.sync()                                   # the rows are produced on the context's stream
            return fn()
        with torch.cuda.stream(self.stream):             # NCCL's stream waits for an event of the current stream
            return fn()

    def _complete(self, work):
        import torch
        if self.stream is None or _TRACE["on"]:
            work.wait()
            torch.cuda.current_stream().synchronize()
            return
        with torch.cuda.stream(self.stream):             # the context's stream waits for the collective; the host goes on
            work.wait()

    def all_to_all_rows_start(self, ctx, send, send_counts, recv_counts):
        """send: DeviceArray whose rows are grouped by destination rank in rank order.  Starts the NCCL all-to-all (over
        NVLink, on torch's NCCL stream) and returns (recv, work): recv holds the rows of rank 0, 1, ... in that order
        once all_to_all_rows_wait(work) has returned; `send` must stay alive until then."""
        w = send.width
        recv = ctx.alloc(sum(recv_counts), w)
        if not self.dist:
            raise RuntimeError("all_to_all on a single rank")
        if _TRACE["on"]:
            ctx.sync()
            self._a2a_t0, self._a2a_bytes = _time.perf_counter(), sum(send_counts) * w
        if isinstance(send, _Repeated):                  # the same rows to every peer (all-gather with uneven sizes)
            st, rt = self._tensor(send.arr), self._tensor(recv)
            roffs = [sum(recv_counts[:d]) * w for d in range(self.world)]
            outs = [rt[roffs[d]:roffs[d] + recv_counts[d] * w] for d in range(self.world)]
            work = self._issue(ctx, lambda: self.dist.all_to_all(outs, [st] * self.world, async_op=True))
            return recv, work
        rt, st = self._tensor(recv), self._tensor(send)
        work = self._issue(ctx, lambda: self.dist.all_to_all_single(rt, st, [c * w for c in recv_counts],
                                                                     [c * w for c in send_counts], async_op=True))
        return recv, work

    def all_to_all_rows_wait(self, work):
        self._complete(work)
        if _TRACE["on"] and self.rank == 0 and getattr(self, "_a2a_t0", None) is not None:
            _TRACE["log"].append(("a2a %.2f GB sent" % (self._a2a_bytes / 1e9), round((_time.perf_counter() - self._a2a_t0) * 1e3, 2)))
            self._a2a_t0 = None

    def all_to_all_rows(self, ctx, send, send_counts, recv_counts):
        recv, work = self.all_to_all_rows_start(ctx, send, send_counts, recv_counts)
        self.all_to_all_rows_wait(work)
        return recv

    # NCCL's send/recv kernels move 16 bytes per thread only between 16-byte aligned pointers; the per-peer segments
    # of a table of 113-byte rows start anywhere, and such an exchange runs at less than half the speed (measured:
    # 11.3 GB per rank in 32 ms against 13.6 ms).  The large exchanges therefore go through byte buffers whose
    # segments start at multiples of 128 bytes on both sides (uqb_gather_rows_segmented / uqb_compact_segments).
    def exchange_rows_start(self, ctx, table, router, send_counts, recv_counts, count_table=None):
        """the rows of `table`, grouped by destination through `router` (see _segmented; send_counts rows each), leave for
        their ranks.  Returns a handle for exchange_rows_wait, which yields the DeviceArray of the rows received from
        rank 0, 1, ... in that order.  With a peer window (and the full count table) the rows are stored straight into
        the receivers' memory by this rank's own kernel; otherwise NCCL moves them."""
        w = table.width
        plan = _p2p_plan(self, ctx, table, router, count_table)
        if plan is not None:
            return _p2p_exchange(self, ctx, table, router, send_counts, recv_counts, plan)
        send_pad, soffs = _segmented(ctx, table, router, send_counts, 128)
        roffs, total = [], 0
        for c in recv_counts:
            roffs.append(total)
            total = (total + c * w + 127) // 128 * 128
        recv_pad = ctx.alloc(total, 1)
        if _TRACE["on"]:
            ctx.sync()
            self._a2a_t0, self._a2a_bytes = _time.perf_counter(), sum(send_counts) * w
        st, rt = self._tensor(send_pad), self._tensor(recv_pad)
        ins = [st[soffs[d]:soffs[d] + send_counts[d] * w] for d in range(self.world)]
        outs = [rt[roffs[d]:roffs[d] + recv_counts[d] * w] for d in range(self.world)]
        work = self._issue(ctx, lambda: self.dist.all_to_all(outs, ins, async_op=True))
        return dict(work=work, send=send_pad, recv=recv_pad, roffs=roffs, recv_counts=list(recv_counts), width=w)

    def exchange_rows_wait(self, ctx, ex):
        if ex.get("p2p"):
            self.window.barrier()                        # every rank's rows have landed
            return ex["recv"]
        self.all_to_all_rows_wait(ex["work"])
        ex["send"].free()
        out = ctx.compact_segments(ex["recv"], ex["roffs"], ex["recv_counts"], ex["width"])
        ex["recv"].free()                                # stream ordered: the copy above is queued before any reuse
        return out

    def barrier(self):
        if self.dist:
            self.dist.barrier(group=self.obj_group)

    def all_gather_rows(self, ctx, local, counts):
        """every rank contributes `local` (counts[rank] rows) -> DeviceArray with the rows of rank 0, 1, ... in that
        order on every rank (the unique tables of the sharded decode).  One all-to-all in which every rank sends its
        rows to everybody: per-peer sizes may differ, which NCCL's all-gather does not allow."""
        if not self.dist:
            return local
        return self.all_to_all_rows(ctx, _Repeated(local, self.world), [local.n] * self.world, list(counts))


class _Repeated:
    """send buffer of an all-to-all in which every peer receives the same rows"""

    def __init__(self, arr, times):
        self.arr, self.times, self.width = arr, times, arr.width


# ------------------------------------------------------------------------------------------------
# W ranks on ONE device (SURVEY section 4d): every rank is a host thread with its own context (stream, arena); the
# collectives are barriers over shared Python slots and device->device copies out of the peers' buffers.  Everything
# else - uqb_partition_positions, the segmented exchange buffers, uqb_compact_segments, the merges, global_order - is the
# code the NCCL ranks run, so the single-GPU test box exercises the whole sharded path.
# ------------------------------------------------------------------------------------------------
class LocalGroup:
    def __init__(self, world):
        import threading
        self.world = world
        self.barrier = threading.Barrier(world)
        self.slots = [None] * world


class LocalComm:
    dist = None

    def __init__(self, group, rank):
        self.group, self.rank, self.world = group, rank, group.world

    def barrier(self):
        self.group.barrier.wait(timeout=600)

    def all_gather_object(self, obj):
        g = self.group
        g.slots[self.rank] = obj
        self.barrier()
        out = list(g.slots)
        self.barrier()
        return out

    def exchange_counts(self, send_counts):
        table = self.all_gather_object(list(map(int, send_counts)))
        return [table[src][self.rank] for src in range(self.world)]

    def _pull(self, ctx, recv, roffs, my_ptr, my_soffs, my_sbytes):
        """recv[roffs[src] ...] <- the bytes rank `src` holds for this rank, for every src"""
        ctx.sync()                                       # my own send buffer is final
        infos = self.all_gather_object((int(my_ptr or 0), list(my_soffs), list(my_sbytes)))
        for src in range(self.world):
            ptr, soffs, sbytes = infos[src]
            if sbytes[self.rank]:
                ctx.copy_in(recv, roffs[src], ptr + soffs[self.rank], sbytes[self.rank])
        ctx.sync()
        self.barrier()                                   # nobody releases its send buffer before every peer has copied

    def all_to_all_rows_start(self, ctx, send, send_counts, recv_counts):
        w = send.width
        recv = ctx.alloc(sum(recv_counts), w)
        if isinstance(send, _Repeated):
            ptr, soffs = send.arr.device_ptr.value, [0] * self.world
        else:
            ptr, soffs = send.device_ptr.value, [sum(send_counts[:d]) * w for d in range(self.world)]
        roffs = [sum(recv_counts[:d]) * w for d in range(self.world)]
        self._pull(ctx, recv, roffs, ptr, soffs, [c * w for c in send_counts])
        return recv, None

    def all_to_all_rows_wait(self, work):
        pass

    def all_to_all_rows(self, ctx, send, send_counts, recv_counts):
        return self.all_to_all_rows_start(ctx, send, send_counts, recv_counts)[0]

    window = None

    def open_window(self, ctx, nbytes, slots=3):
        """the emulated ranks share one device: every rank's buffer is directly addressable by the others"""
        buf = ctx.alloc(int(nbytes), 1)
        ptrs = self.all_gather_object(int(buf.device_ptr.value))

        def barrier():
            ctx.sync()
            self.barrier()
        self.window = PeerWindow(ptrs, self.rank, int(nbytes), slots, barrier, keep=buf)

    def exchange_rows_start(self, ctx, table, router, send_counts, recv_counts, count_table=None):
        w = table.width
        plan = _p2p_plan(self, ctx, table, router, count_table)
        if plan is not None:
            return _p2p_exchange(self, ctx, table, router, send_counts, recv_counts, plan)
        send_pad, soffs = _segmented(ctx, table, router, send_counts, 128)
        roffs, total = [], 0
        for c in recv_counts:
            roffs.append(total)
            total = (total + c * w + 127) // 128 * 128
        recv_pad = ctx.alloc(total, 1)
        self._pull(ctx, recv_pad, roffs, send_pad.device_ptr.value, soffs, [c * w for c in send_counts])
        return dict(work=None, send=send_pad, recv=recv_pad, roffs=roffs, recv_counts=list(recv_counts), width=w)

    def exchange_rows_wait(self, ctx, ex):
        if ex.get("p2p"):
            self.window.barrier()
            return ex["recv"]
        ex["send"].free()
        out = ctx.compact_segments(ex["recv"], ex["roffs"], ex["recv_counts"], ex["width"])
        ex["recv"].free()
        return out

    def all_gather_rows(self, ctx, local, counts):
        return self.all_to_all_rows(ctx, _Repeated(local, self.world), [local.n] * self.world, list(counts))


def run_local(world, fn, device=0):
    """Run fn(ctx, comm) on `world` emulated ranks of one device (one host thread and one context per rank).
    -> [fn's result per rank]; the first exception of any rank is re-raised after all threads have stopped."""
    import threading
    from .device import Context
    group = LocalGroup(world)
    results, errors = [None] * world, [None] * world
    create = threading.Lock()

    def body(rank):
        ctx = None
        try:
            with create:                                 # library start-up (driver entry points) is not re-entrant
                ctx = Context(device)
            results[rank] = fn(ctx, LocalComm(group, rank))
        except BaseException as e:                       # noqa: a failed rank must release the others
            errors[rank] = e
            group.barrier.abort()
        finally:
            if ctx is not None:
                try:
                    ctx.sync()
                    ctx.close()
                except Exception:
                    pass

    threads = [threading.Thread(target=body, args=(r,), daemon=True) for r in range(world)]
    for t in threads: t.start()
    for t in threads: t.join()
    import threading as _t
    real = [e for e in errors if e is not None and not isinstance(e, _t.BrokenBarrierError)]
    if real:
        raise real[0]
    if any(errors):
        raise [e for e in errors if e is not None][0]
    return results


# ------------------------------------------------------------------------------------------------
# distributed sort / unique
# ------------------------------------------------------------------------------------------------
SAMPLES_PER_RANK = 1024
SKEW_LIMIT = 2.0          # a rank may receive at most this many times the largest local table, else the merge variant runs


def row_key64(rows):
    """uint8 [m][w] -> uint64: the first 8 bytes of every row as a big-endian integer (zero padded) - the partition key"""
    m, w = rows.shape
    buf = np.zeros((m, 8), dtype=np.uint8)
    buf[:, :min(8, w)] = rows[:, :8]
    return buf.view(">u8").reshape(-1).astype(np.uint64)


def _sample_rows(ctx, table, count):
    n, w = table.n, table.width
    if n == 0:
        return np.zeros((0, w), dtype=np.uint8)
    idx = np.unique(np.linspace(0, n - 1, num=min(n, count)).astype(np.uint32))
    d_idx = ctx.upload(idx)
    d_s = ctx.gather_rows(table, d_idx)
    out = d_s.download().reshape(len(idx), w) if w else np.zeros((len(idx), 0), np.uint8)
    d_idx.free(); d_s.free()
    return out


def global_unique(ctx, comm, table, want_perm=False):
    """-> dict(key: uint32[n] global unique-row index of every local row, uniq: this rank's key range of the global
    unique table (rows ascending; the ranges concatenate in rank order), n_unique, counts (unique rows per rank),
    route: how to bring per-record arrays into the global stable order of this table (see global_order)).

    Partition first, sort once: splitters come from a sample of every rank's rows; a row goes to the rank whose range
    holds its first 8 bytes (so identical rows, and all rows tied on those bytes, meet on one rank); ONE all-to-all
    moves the rows over NVLink, each rank sorts / uniques its range exactly like the single-GPU path, and the global
    ids travel back through the reverse all-to-all.  If the sample is fooled by a very skewed table (one rank would
    receive more than SKEW_LIMIT times the largest local table) the merge variant below runs instead.

    global_unique_begin / global_unique_end are the two halves around the row exchange: encode_sharded starts the
    exchange of one table and prepares or finishes another one while the rows are on the wire."""
    return global_unique_end(ctx, comm, global_unique_begin(ctx, comm, table, want_perm=want_perm))


def gather_samples(ctx, comm, tables):
    """row samples of several tables in ONE collective -> {name: what global_unique_begin(gathered=...) expects}"""
    mine = {t: (_sample_rows(ctx, a, SAMPLES_PER_RANK), a.n) for t, a in tables.items()}
    parts = comm.all_gather_object(mine)
    return {t: [p[t] for p in parts] for t in tables}


def global_unique_begin(ctx, comm, table, want_perm=False, gathered=None):
    if comm.world == 1:
        perm, key_local, uniq_local, nu = ctx.sort_rows(table, want_perm=want_perm, want_key=True, want_uniq=True)
        return dict(done=dict(key=key_local, uniq=uniq_local, n_unique=nu, counts=[nu], route=("local", perm)))
    _mark(ctx, comm, None)
    if gathered is None:
        samples = _sample_rows(ctx, table, SAMPLES_PER_RANK)
        gathered = comm.all_gather_object((samples, table.n))
    _mark(ctx, comm, "gu.sample")
    splitters = pick_splitters(np.concatenate([g[0] for g in gathered]), comm.world)
    pos, send_counts = ctx.partition_positions(table, np.sort(row_key64(splitters)))      # one sequential sweep
    router = [pos]
    send_counts += [0] * (comm.world - len(send_counts))
    count_table = comm.all_gather_object(list(map(int, send_counts)))            # one collective: who sends how much to whom
    recv_counts = [count_table[src][comm.rank] for src in range(comm.world)]
    worst = max(sum(count_table[src][dst] for src in range(comm.world)) for dst in range(comm.world))
    _mark(ctx, comm, "gu.partition")
    if worst > SKEW_LIMIT * max(g[1] for g in gathered) + 4096 or os.environ.get("UQB_MG_MERGE") == "1":
        _router_free(router)
        return dict(done=global_unique_merge(ctx, comm, table, want_perm=want_perm))
    ex = comm.exchange_rows_start(ctx, table, router, send_counts, recv_counts, count_table=count_table)
    recv = None
    if _TRACE["on"]:                                     # diagnostics: time the exchange on its own (no overlap)
        recv = comm.exchange_rows_wait(ctx, ex)
        _mark(ctx, comm, "gu.exchange(sync)")
    return dict(done=None, ex=ex, recv=recv, router=router, send_counts=send_counts, recv_counts=recv_counts, want_perm=want_perm,
                count_table=count_table)


def global_unique_end(ctx, comm, st):
    if st["done"] is not None:
        return st["done"]
    _mark(ctx, comm, None)
    recv = st["recv"] if st["recv"] is not None else comm.exchange_rows_wait(ctx, st["ex"])
    _mark(ctx, comm, "gu.exchange_wait")
    router, send_counts, recv_counts, want_perm = st["router"], st["send_counts"], st["recv_counts"], st["want_perm"]
    if want_perm:
        # The sorted-on table: the records are going to follow their rows to this rank anyway (global_order), so the key of
        # this rank's slice of the global order is the group id in SORTED order - no trip back to the record's rank and
        # forth again.
        perm_r, _, uniq_range, nr, key_sorted = ctx.sort_rows(recv, want_perm=True, want_uniq=True, want_key_sorted=True)
        recv.free()
        _mark(ctx, comm, "gu.sort")
        counts = comm.all_gather_object(nr)
        ctx.add_scalar_u32(key_sorted, sum(counts[:comm.rank]))
        route = ("partition", router, send_counts, recv_counts, perm_r, st["count_table"])
        return dict(key=None, key_sorted=key_sorted, uniq=uniq_range, n_unique=sum(counts), counts=counts, route=route)
    _, key_r, uniq_range, nr = ctx.sort_rows(recv, want_key=True, want_uniq=True)
    recv.free()
    _mark(ctx, comm, "gu.sort")
    counts = comm.all_gather_object(nr)
    ctx.add_scalar_u32(key_r, sum(counts[:comm.rank]))       # global id of every received row
    ids_back = comm.all_to_all_rows(ctx, key_r, recv_counts, send_counts)        # in the order the rows were sent
    key_r.free()
    # ids_back is in the order the rows were sent: row i was sent at position pos[i]
    key_global = ctx.gather_rows(ids_back, router[0])
    ids_back.free()
    _mark(ctx, comm, "gu.ids_back")
    _router_free(router)
    return dict(key=key_global, uniq=uniq_range, n_unique=sum(counts), counts=counts, route=None)


def global_unique_merge(ctx, comm, table, want_perm=False):
    """The merge variant: every rank sorts / uniques its own rows first, only the locally unique rows travel, and the
    receiving rank sorts them again.  Twice the sorting, but immune to skew (a table of identical rows sends one row)."""
    perm, key_local, uniq_local, nu = ctx.sort_rows(table, want_perm=want_perm, want_key=True, want_uniq=True)
    w = table.width
    samples = _sample_rows(ctx, uniq_local, 256)
    splitters = pick_splitters(np.concatenate(comm.all_gather_object(samples)), comm.world)
    if len(splitters) == comm.world - 1:
        b = [0] + [int(x) for x in ctx.rows_lower_bound(uniq_local, splitters)] + [nu]
        for i in range(1, len(b)):                      # equal splitters give equal bounds; keep them monotone
            b[i] = max(b[i], b[i - 1])
    else:                                               # nothing anywhere
        b = [0] * comm.world + [nu]
    send_counts = [b[k + 1] - b[k] for k in range(comm.world)]
    recv_counts = comm.exchange_counts(send_counts)
    recv = comm.all_to_all_rows(ctx, uniq_local, send_counts, recv_counts)
    uniq_local.free()
    _, key_recv, uniq_range, nr = ctx.sort_rows(recv, want_key=True, want_uniq=True)
    recv.free()
    counts = comm.all_gather_object(nr)
    offset = sum(counts[:comm.rank])
    ctx.add_scalar_u32(key_recv, offset)                # global id of every received unique row
    ids_back = comm.all_to_all_rows(ctx, key_recv, recv_counts, send_counts)     # in the order the rows were sent = sorted
    key_recv.free()
    key_global = ctx.gather_rows(ids_back, key_local)   # ids_back[local unique index]
    ids_back.free(); key_local.free()
    route = ("merge", key_global, perm, counts) if want_perm else None
    return dict(key=key_global, uniq=uniq_range, n_unique=sum(counts), counts=counts, route=route)


def global_order(ctx, comm, route, payloads):
    """Bring per-record arrays into the global stable order of the sorted-on table.  payloads: {name: DeviceArray [n][w]}
    -> {name: DeviceArray} holding this rank's slice of the globally sorted arrays (slices concatenate in rank order).
    Frees the route's arrays (not the payloads)."""
    kind = route[0]
    if kind == "local":
        perm = route[1]
        out = {k: ctx.gather_rows(v, perm) for k, v in payloads.items()}
        perm.free()
        return out
    if kind == "partition":
        # the records follow their rows: same partition, same all-to-all, then the receiving rank's stable argsort.
        # Source ranks arrive in rank order and every source keeps its record order, so ties end in global record order.
        _, router, send_counts, recv_counts, perm_r, count_table = route
        out = {}
        pending = None
        for name, arr in payloads.items():               # the exchange of one array overlaps the final gather of the previous one
            ex = comm.exchange_rows_start(ctx, arr, router, send_counts, recv_counts, count_table=count_table)
            if pending is not None:
                out[pending[0]] = ctx.gather_rows(pending[1], perm_r)
                pending[1].free()
            pending = (name, comm.exchange_rows_wait(ctx, ex))
        if pending is not None:
            out[pending[0]] = ctx.gather_rows(pending[1], perm_r)
            pending[1].free()
        _router_free(router); perm_r.free()
        _mark(ctx, comm, "global_order")
        return out
    _, key_global, perm, counts = route
    # merge variant: every record goes to the rank that owns its key range; there a stable sort by key finishes the job
    key_sorted = ctx.gather_rows(key_global, perm)                      # non-decreasing
    key_be = ctx.columns_to_rows([key_sorted])                          # big-endian rows: memcmp order = numeric order
    bounds = np.cumsum(counts)[:-1].astype(">u4").view(np.uint8).reshape(-1, 4)
    b = [0] + [int(x) for x in ctx.rows_lower_bound(key_be, bounds)] + [key_sorted.n]
    key_be.free()
    send_counts = [b[k + 1] - b[k] for k in range(comm.world)]
    recv_counts = comm.exchange_counts(send_counts)
    key_recv = comm.all_to_all_rows(ctx, key_sorted, send_counts, recv_counts)
    key_sorted.free()
    kb = ctx.columns_to_rows([key_recv])
    perm2, _, _, _ = ctx.sort_rows(kb, want_perm=True)                  # stable
    kb.free(); key_recv.free()
    out = {}
    for name, arr in payloads.items():
        s = ctx.gather_rows(arr, perm)
        r = comm.all_to_all_rows(ctx, s, send_counts, recv_counts)
        s.free()
        out[name] = ctx.gather_rows(r, perm2)
        r.free()
    perm2.free(); perm.free()
    return out


# ------------------------------------------------------------------------------------------------
# the encode
# ------------------------------------------------------------------------------------------------
class ShardResult:
    """This rank's part of every member.  `slices[name]` = (DeviceArray, kind, meta):
      kind 'vector'  meta = dtype; the members concatenate over the ranks in rank order
      kind 'table'   meta = dict(width, pattern, rows): the DeviceArray holds the byte stream of this rank's `rows`
                     logical rows under `pattern` (uqb_layout of the local rows).  Where those bytes sit in the
                     member's global stream follows from the pattern (place()): row-major streams are one byte range
                     (counted from the other end when the pattern reverses the rows), column-major streams one run of
                     `rows` bytes per byte column at col * N + first row (SURVEY section 8e, "layout").
    place(comm) adds the global geometry (first row of this rank, total rows) with one small object collective."""

    def __init__(self, ctx=None, sink=None):
        self.slices = {}
        self.ctx, self.sink, self.host = ctx, sink, {}
        self.geometry = {}          # name -> (first logical row / element of this rank, total over the ranks)

    def add(self, name, arr, kind, meta):
        """with a sink ((name, nbytes) -> pinned uint8 ndarray) the device->host copy starts right away"""
        self.slices[name] = (arr, kind, meta)
        if self.sink is not None:
            buf = self.sink(name, arr.nbytes)
            arr.download_async(buf)
            self.host[name] = buf

    def rows_of(self, name):
        arr, kind, meta = self.slices[name]
        return meta['rows'] if kind == 'table' else arr.n

    def place(self, comm):
        mine = {name: self.rows_of(name) for name in self.slices}
        allr = comm.all_gather_object(mine)
        for name in self.slices:
            per = [a[name] for a in allr]
            self.geometry[name] = (sum(per[:comm.rank]), sum(per))

    def nbytes(self):
        return sum(a.nbytes for a, _, _ in self.slices.values())

    def download(self):
        """-> {name: flat uint8 ndarray (tables: the local stream) or typed 1-D ndarray (vectors)}"""
        out = {}
        if self.sink is not None:
            self.ctx.copy_sync()
        for name, (arr, kind, meta) in self.slices.items():
            flat = self.host[name][:arr.nbytes] if self.sink is not None else arr.download(dtype=np.uint8).reshape(-1)
            out[name] = flat.view(np.dtype(meta)).reshape(-1) if kind == "vector" else flat
        return out

    def describe(self):
        """picklable description of this rank's slices: name -> (kind, meta, first, total)"""
        return {name: (kind, str(np.dtype(meta)) if kind == 'vector' else dict(meta)) + self.geometry[name]
                for name, (_, kind, meta) in self.slices.items()}

    def free(self):
        if self.sink is not None and self.ctx is not None:
            self.ctx.copy_sync()
        for arr, _, _ in self.slices.values():
            arr.free()
        self.slices = {}

    def __del__(self):
        try:
            if self.slices and self.ctx is not None and self.ctx.h:
                self.free()             # queued device->host copies must finish before the arrays are recycled
        except Exception:
            pass


def place_slice(dst_flat, kind, meta, first, total, data):
    """Put one rank's slice `data` (flat bytes / typed vector) into the member's global buffer `dst_flat`."""
    if kind == 'vector':
        dst_flat[first:first + len(data)] = data
        return
    width, pattern, rows = meta['width'], meta['pattern'], meta['rows']
    transposed, rev_r, _ = host.PATTERN_DESC[pattern]
    at = total - first - rows if rev_r else first
    if not transposed:
        dst_flat[at * width:(at + rows) * width] = data
    else:
        dst_flat.reshape(width, total)[:, at:at + rows] = data.reshape(width, rows)


def encode_sharded(ctx, comm, fq, sort=None, raw=None, pattern=None, pad=False, notricks=False, sink=None):
    """fq: this rank's contiguous range of the reads (device.Fastq).  -> (ShardResult, config); config is identical on
    every rank and equal to the single-GPU config of the whole file."""
    sort, raw, pattern = host.normalise_options(sort, raw, pattern)
    pat_of = {'DNA': pattern[0], 'QUAL': pattern[1]}
    _mark(ctx, comm, None)
    info = fq.split()
    n_local = int(info.n_reads)
    lines_bad = info.status == 1
    counts = comm.all_gather_object((n_local, lines_bad))
    if any(b for _, b in counts):
        raise host.UQError('ERROR: The FASTQ file provided contains a number of rows which is not divisible by 4!')
    ns = [c for c, _ in counts]
    n_total = sum(ns)
    base = sum(ns[:comm.rank])
    if n_total == 0:
        raise host.UQError('ERROR: the FASTQ file holds no records')
    if any(c == 0 for c in ns):
        raise host.UQError('ERROR: every rank needs at least one read')
    if n_total > 10000 and ns[0] < 10001:
        raise host.UQError('ERROR: rank 0 must hold the first 10001 reads (Pass-2 checkpoint 0)')
    # ---- Pass 1 against the global first QNAME line ----
    first_off = fq.line_offsets(0, 2)
    my_first = fq.download(0, int(first_off[1]) - 1).tobytes()
    ref = comm.all_gather_object(my_first)[0]
    if fq.reference != ref:                            # a streamed load may already have measured against it
        fq.set_reference(ref, base)
    plain = stats_to_plain(fq.analyze())
    parts = comm.all_gather_object((plain, base, n_local))
    parts[0][0]["first_name"] = ref
    st = merge_stats(parts)
    if st.bad_first_char != -1:
        raise host.UQError('ERROR: This does not look like a FASTA/FASTQ file! (first line does not start with @)')
    bad = [(r, w) for r, w in ((st.bad_plus_record, 'plus'), (st.bad_len_record, 'len')) if r >= 0]
    if bad:
        r, w = min(bad, key=lambda t: (t[0], t[1] != 'plus'))
        raise host.UQError('ERROR: malformed FASTQ record %d (%s)' % (r, w))
    dec = host.decide_alphabets(st, notricks=notricks, pad=pad)
    _mark(ctx, comm, "split+pass1")
    # ---- Pass 2: rank 0 decides which columns leave 'mapping' at checkpoint 0, the others skip those dictionaries ----
    pass2_of = {}                                   # this rank's and the merged dictionaries of the final layout

    def scan(prefix, suffix, separators):
        """column statistics of the whole file; a record that does not split on ANY rank switches every rank to E2"""
        ncols = len(separators) + 1
        # which columns leave 'mapping' at checkpoint 0 is a property of the first 10001 records of the file: rank 0
        # scans just that head (a few megabytes) and tells the others, then every rank scans its own range at the same time
        early = None
        if comm.rank == 0:
            early = [False] * ncols
            if n_total > 10000:
                head_bytes = int(fq.line_offsets(4 * 10001, 1)[0])
                hfq = ctx.load_fastq(fq.download(0, head_bytes))
                hfq.split()
                hcols, hbad = hfq.qname_scan(len(prefix), len(suffix), separators)
                if hbad < 0:
                    early = [bool(hcols[c].n_distinct == L.U64_MAX) for c in range(ncols)]
                hfq.free()
        early = comm.all_gather_object(early)[0]
        cols0, bad0 = fq.qname_scan(len(prefix), len(suffix), separators, col_mode=[1 if e else 2 for e in early])
        my_dicts = {}
        if bad0 < 0:
            for c in range(ncols):
                if not early[c]:
                    toks = fq.qname_dict(c)
                    my_dicts[c] = (toks, (fq.qname_dict_first(c).astype(np.int64) + base).tolist())
        pass2 = comm.all_gather_object((bad0, colstats_to_plain(cols0, ncols) if bad0 < 0 else None, my_dicts))
        bad = [base_r + p[0] for p, (_, base_r, _) in zip(pass2, parts) if p[0] >= 0]
        if bad:
            return None, min(bad)
        colstats, merged = merge_colstats([p[1] for p in pass2], n_total, early, [p[2] for p in pass2])
        pass2_of.update(local=my_dicts, merged=merged)
        return colstats, -1

    def shortest_remainder(plen):
        cols, _ = fq.qname_scan(plen, 0, '', col_mode=[1])
        return min(comm.all_gather_object(int(cols[0].min_len)))

    prefix, suffix, separators, columns = host.decide_qname_columns(st, n_total, scan, shortest_remainder,
                                                                    lambda i: pass2_of['merged'][i])
    my_dicts, gdicts = pass2_of['local'], pass2_of['merged']
    _mark(ctx, comm, "pass2")
    # ---- pack + column encode (per read) ----
    dna, qual = fq.pack(host.pack_params(dec))
    specs = host.column_specs(columns)
    cols = fq.qname_encode([(f, 4 if f == 0 else size, off, mn) for f, size, off, mn in specs])
    for c, meta in enumerate(columns):
        if meta['format'] == 'mapping':                 # local dictionary rank -> global dictionary rank
            local = my_dicts[c][0]
            remap = np.searchsorted(np.array(gdicts[c], dtype=object), np.array(local, dtype=object)).astype(np.uint32) if local else np.zeros(0, np.uint32)
            d_remap = ctx.upload(remap)
            g = ctx.gather_rows(d_remap, cols[c])
            d_remap.free(); cols[c].free()
            cols[c] = ctx.narrow_u32(g, specs[c][1])
            g.free()
    _mark(ctx, comm, "pack+cols")
    # ---- run_mix over the ranks ----
    res = ShardResult(ctx, sink)

    def add_table(name, rows_arr, t):
        """this rank's rows of a DNA / QUAL member -> their stream under the table's --pattern (uq.py:257-270)"""
        pat = pat_of[t]
        if pat == '0.1':
            stream = rows_arr
        else:
            stream = ctx.layout(rows_arr, pat)
            rows_arr.free()
        res.add(name, stream, 'table', dict(width=rows_arr.width, pattern=pat, rows=rows_arr.n))

    sorted_on = sort if sort in ('DNA', 'QUAL', 'QNAME') else None
    # QNAME keeps its sort rows here, not the packed key of host.qname_sort_table: the sample-sort partition and the
    # splitter search read row bytes
    tables = {'DNA': dna, 'QUAL': qual, 'QNAME': host.qname_rows(ctx, cols, columns)}
    keyed = {t: (t not in raw) for t in tables}
    uniq = {}
    payload = {}
    in_order = {}                                   # arrays that are produced in the global order (no global_order trip)
    route = None
    for t in ('DNA', 'QUAL', 'QNAME'):
        if not keyed[t]:
            if t == 'QNAME':
                for c, meta in zip(cols, columns):
                    payload[meta['name'] + '.raw'] = c
            else:
                payload[t + '.raw'] = tables[t]

    def finish(t, st):
        nonlocal route
        g = global_unique_end(ctx, comm, st)
        if t == sorted_on:
            route = g['route']
        if keyed[t]:
            uniq[t] = (g['uniq'], g['n_unique'])
            if g.get('key_sorted') is not None:     # already this rank's slice of the global order
                in_order[t + '.key'] = g['key_sorted']
            else:
                payload[t + '.key'] = g['key']
            if t == 'QNAME':                        # unique rows back to typed columns (uq.py:842-847)
                ucols = host.qname_columns(ctx, g['uniq'], columns, None)
                for c, meta in zip(ucols, columns):
                    res.add(meta['name'], c, 'vector', meta['dtype'])
                g['uniq'].free()
            else:
                add_table(t, g['uniq'], t)
        else:
            g['uniq'].free()
            if g.get('key_sorted') is not None:
                g['key_sorted'].free()
            elif not (t == sorted_on and route[0] == 'merge'):      # the merge route still needs the key
                g['key'].free()

    # software pipeline over the tables: while the rows of one table are on the wire (NCCL stream), the next table is
    # sampled / partitioned / gathered and the previous one is sorted (context stream).  DNA goes first: its exchange is
    # the shortest one to leave uncovered, and the long QUAL exchange then hides behind the DNA sort.
    todo = [t for t in ('DNA', 'QUAL', 'QNAME') if keyed[t] or t == sorted_on]
    samples = gather_samples(ctx, comm, {t: tables[t] for t in todo}) if comm.world > 1 and todo else {}
    pending = None
    for t in todo:
        st = global_unique_begin(ctx, comm, tables[t], want_perm=(t == sorted_on), gathered=samples.get(t))
        if pending is not None:
            finish(*pending)
        pending = (t, st)
    if pending is not None:
        finish(*pending)
    if route is not None:
        moved = global_order(ctx, comm, route, payload)
        old = {id(v): v for v in payload.values()}
        if route[0] == 'merge':
            old[id(route[1])] = route[1]
        for v in old.values():
            v.free()
        payload = moved
    payload.update(in_order)
    # keys are narrowed to min_scalar_type(max(key)) of the WHOLE file (uq.py:790, 832)
    for t in ('DNA', 'QUAL', 'QNAME'):
        if keyed[t]:
            u, nu = uniq[t]
            size = host.key_itemsize(nu)
            k32 = payload[t + '.key']
            res.add(t + '.key', ctx.narrow_u32(k32, size), 'vector', 'uint%d' % (8 * size))
        elif t == 'QNAME':
            for meta in columns:
                res.add(meta['name'] + '.raw', payload[meta['name'] + '.raw'], 'vector', meta['dtype'])
        else:
            add_table(t + '.raw', payload[t + '.raw'], t)
    if tables['QNAME'] is not None:
        tables['QNAME'].free()
    res.place(comm)
    return res, host.config_of(dec, n_total, prefix, suffix, separators, columns, sort, raw, pattern)


def assemble(comm, res):
    """Gather every rank's host slices on rank 0 and put them at their place in the global members -> members dict
    (name -> ndarray as numpy.save would receive it) on rank 0, None elsewhere.  Test / small-file helper: the container
    writer (write_container_sharded below) lets every rank write its slices at their byte offsets of the tar instead."""
    parts = comm.all_gather_object((res.describe(), res.download()))
    if comm.rank != 0:
        return None
    out = {}
    for name, (kind, meta, _, total) in parts[0][0].items():
        if kind == 'vector':
            flat = np.empty(total, dtype=np.dtype(meta))
        else:
            flat = np.empty(total * meta['width'], dtype=np.uint8)
        for desc, data in parts:
            k, m, first, tot = desc[name]
            place_slice(flat, k, m, first, tot, data[name])
        out[name] = flat if kind == 'vector' else host.table_ndarray(flat, total, meta['width'], meta['pattern'])
    return out


def write_container_sharded(comm, path, res, config):
    """ONE container file written by all ranks (SURVEY section 8 f2): rank 0 plans the byte layout from the global
    shapes and writes the tar / NPY headers and config.json, then every rank puts its slices at their byte offsets
    with pwrite - vectors and row-major streams as one range, column-major streams as one run per byte column.
    `path` must be reachable by every rank (one node).  The file is byte-identical to the single-GPU container."""
    from . import container
    desc = res.describe()
    data = res.download()
    offsets = None
    if comm.rank == 0:
        entries = {}
        for name, (kind, meta, _, total) in desc.items():
            if kind == 'vector':
                entries[name] = (np.dtype(meta), (total,), False)
            else:
                w, pat = meta['width'], meta['pattern']
                shape = (total, w) if pat[0] in '02' else (w, total)
                entries[name] = (np.uint8, shape, pat[2] == '2' and total > 1 and w > 1)     # numpy writes both-contiguous arrays as C
        plan = container.Plan(entries, config)
        plan.create(path)
        offsets = plan.offsets
    offsets = comm.all_gather_object(offsets)[0]             # doubles as the barrier behind the file's creation
    fd = os.open(path, os.O_WRONLY)
    try:
        for name, (kind, meta, first, total) in desc.items():
            base = offsets[name][1]
            buf = data[name]
            if kind == 'vector':
                container._pwrite_all(fd, buf.view(np.uint8), base + first * buf.dtype.itemsize)
                continue
            width, pattern, rows = meta['width'], meta['pattern'], meta['rows']
            transposed, rev_r, _ = host.PATTERN_DESC[pattern]
            at = total - first - rows if rev_r else first
            if not transposed:
                container._pwrite_all(fd, buf, base + at * width)
            else:
                for col in range(width):
                    container._pwrite_all(fd, buf[col * rows:(col + 1) * rows], base + col * total + at)
    finally:
        os.close(fd)
    comm.barrier()


# ------------------------------------------------------------------------------------------------
# the decode (uq.py:926-1060) over the ranks: every rank produces the text of a contiguous range of records
# ------------------------------------------------------------------------------------------------
def split_evenly(n_total, rank, world):
    base, rem = divmod(n_total, world)
    first = rank * base + min(rank, rem)
    return first, first + base + (1 if rank < rem else 0)


def decode_sharded(ctx, comm, members, config):
    """members / config as container.read_container returns them (every rank can read the container) -> (text, first,
    last): uint8 ndarray with the FASTQ text of records [first, last) of the file; the texts concatenate in rank order.

    Raw tables: a rank uploads only the part of the member's stream that holds its rows (host.stream_rows) and undoes
    the layout on the device.  Keyed tables: every rank uploads 1/W of the unique table, the shares are all-gathered
    over NVLink (all_gather_rows; they are the small side of a keyed container), and the rank's slice of the key
    selects its rows (SURVEY section 8e, "decode")."""
    n = int(config['reads'])
    a, b = split_evenly(n, comm.rank, comm.world)
    pat = config['pattern']

    def upload_rows(arr, pattern, r0, r1):
        width = arr.shape[1] if pattern[0] in '02' else arr.shape[0]
        stream = ctx.upload(host.stream_rows(arr, pattern, r0, r1), width=1)
        tab = ctx.unlayout(stream, r1 - r0, width, pattern)
        stream.free()
        return tab

    def table(name, pattern):
        if name + '.raw' in members:
            arr = members[name + '.raw']
            if (arr.shape[0] if pattern[0] in '02' else arr.shape[1]) != n:
                raise host.UQError('ERROR: %s.raw does not hold %d rows' % (name, n))
            return upload_rows(arr, pattern, a, b)
        if name in members and name + '.key' in members:
            arr = members[name]
            u = arr.shape[0] if pattern[0] in '02' else arr.shape[1]
            shares = [split_evenly(u, r, comm.world) for r in range(comm.world)]
            mine = upload_rows(arr, pattern, *shares[comm.rank])
            uniq = comm.all_gather_rows(ctx, mine, [e - s0 for s0, e in shares])
            if uniq is not mine:
                mine.free()
            key = host._upload_key(ctx, members[name + '.key'][a:b], u, name + '.key')
            tab = ctx.gather_rows(uniq, key)
            uniq.free(); key.free()
            return tab
        raise host.UQError('ERROR: No %s data was found in this uQ file?!' % name)

    dna = table('DNA', pat[0])
    qual = table('QUAL', pat[1])
    cols_meta = config['QNAME_columns']
    keyed = 'QNAME.key' in members
    dcols, key = [], None
    for i, meta in enumerate(cols_meta):
        nm = 'QNAME_%d' % (i + 1) + ('' if keyed else '.raw')
        if nm not in members:
            raise host.UQError('ERROR: No QNAME data exists in this uQ file?')
        col = np.ascontiguousarray(members[nm], dtype=meta['dtype'])
        if keyed:
            if key is None:
                key = host._upload_key(ctx, members['QNAME.key'][a:b], len(col), 'QNAME.key')
            c = ctx.upload(col)                       # unique QNAME columns: small, every rank takes them whole
            c2 = ctx.gather_rows(c, key)
            c.free()
            dcols.append(c2)
        else:
            dcols.append(ctx.upload(col[a:b]))
    if key is not None:
        key.free()
    text = host.decode_device(ctx, dna, qual, dcols, config)
    data = text.download().reshape(-1)
    for arr in [dna, qual, text] + dcols:
        arr.free()
    return data, a, b
