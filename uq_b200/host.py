"""Host side of the B200 uQ path: the reference's decision logic re-typed in Python 3 on top of the
statistics the device returns, and the orchestration of the device stages.

Nothing here touches per-read data on the CPU: the FASTQ bytes go to HBM once, every O(N) step is a
call into libuqb200.so (uq_b200/device.py), and what comes back is either O(alphabet) statistics or
the finished output arrays.  There is no CPU fallback and nothing is imported from oracle/.

Reference regions mirrored here (JohnLonginotto/uq, uq.py):
  option validation ............... uq.py:52-69, 893-894          normalise_options
  prefix / suffix / separators .... uq.py:395-413, 427-444        derive_qname_layout
  alphabets, N-trick, bit widths .. uq.py:448-457, 476-545        decide_alphabets
  Pass-2 column typing ............ uq.py:586-602, 641-676        decide_columns
  run_mix / encode_* .............. uq.py:739-851                 run_mix
  config / container .............. uq.py:681-696, 898-912        encode(), container.py
  decoder ......................... uq.py:939-1058                decode()
"""
import re

import numpy as np

from . import _lib as L
from .device import Context, DeviceArray, PATTERN_ID

PATTERNS = ['0.1', '1.1', '2.1', '3.1', '0.2', '1.2', '2.2', '3.2']
# pattern id -> (transposed, rows reversed, bytes reversed) of the byte stream numpy.save emits for the logical table
# m[N][B] (uq.py:263-270, SURVEY A.4): row-major stream[r' * B + b'] or column-major stream[b' * N + r']
PATTERN_DESC = {'0.1': (0, 0, 0), '1.2': (0, 0, 1), '3.2': (0, 1, 0), '2.1': (0, 1, 1),
                '0.2': (1, 0, 0), '1.1': (1, 0, 1), '3.1': (1, 1, 0), '2.2': (1, 1, 1)}
_DT = [(255, 'uint8', 1), (65535, 'uint16', 2), (4294967295, 'uint32', 4), (18446744073709551615, 'uint64', 8)]
STRING_MAX = 255     # widest 'strings' column (E1): uqb_colspec.itemsize / uqb_decode_col.itemsize are uint8


class UQError(Exception):
    """Where the reference prints a message and exit()s (uq.py:48-50) this path raises."""


PHASE_LOG = None     # set to a dict to collect wall-clock milliseconds per phase (adds stream syncs; diagnostics only)
PHASE_KERNELS = None # set to a dict (with the context's kernel timing on) to also collect the kernels of every phase


def _timed(ctx, name, fn, *args, **kw):
    if PHASE_LOG is None:
        return fn(*args, **kw)
    import time
    ctx.sync()
    before = ctx.timing_report() if PHASE_KERNELS is not None else None
    t0 = time.perf_counter()
    out = fn(*args, **kw)
    ctx.sync()
    PHASE_LOG[name] = PHASE_LOG.get(name, 0.0) + (time.perf_counter() - t0) * 1e3
    if before is not None:
        slot = PHASE_KERNELS.setdefault(name, {})
        for k, v in ctx.timing_report().items():
            b = before.get(k, (0, 0.0, 0))
            if v[0] > b[0]:
                c = slot.get(k, (0, 0.0))
                slot[k] = (c[0] + v[0] - b[0], c[1] + v[1] - b[1])
    return out


# ------------------------------------------------------------------------------------------------
# options (uq.py:52-69, 893-894)
# ------------------------------------------------------------------------------------------------
def normalise_options(sort=None, raw=None, pattern=None):
    if pattern is not None:
        if len(pattern) != 2: raise UQError('ERROR: There must be 2 values for --pattern!')
        if not all(p in PATTERNS for p in pattern): raise UQError('ERROR: Pattern values are incorrect!')
    if sort is not None and not isinstance(sort, tuple):
        if sort.lower() not in ('dna', 'qual', 'qname', 'none'): raise UQError('ERROR: --sort value is incorrect!')
        if sort.lower() == 'none': sort = (None,)
    if raw is not None:
        if not all((x is None) or x.lower() in ('dna', 'qual', 'qname', 'none') for x in raw):
            raise UQError('ERROR: --raw values are incorrect!')
        raw = set(raw)
        if 'none' in raw:
            raw.add(None); raw.discard('none')
    if sort is None: sort = (None,)
    if raw is None: raw = (None,)
    if pattern is None: pattern = ['0.1', '0.1']
    return sort, raw, list(pattern)


# ------------------------------------------------------------------------------------------------
# Pass-1 decisions
# ------------------------------------------------------------------------------------------------
def _none(v):
    return v == L.NONE_I64


def derive_qname_layout(st, n_reads):
    """prefix, suffix, ordered separators from the device statistics.

    The reference's loop (uq.py:395-413) is order dependent: a character becomes a separator
    candidate when the running common prefix first shrinks past its last occurrence in line 1, and
    from that record on every QNAME must hold as many of it as line 1.  With
        E[j]  = first record whose common prefix with line 1 is <= j      (from first_lcp_eq)
        M[c]  = last record whose count of c differs from line 1's        (last_count_mismatch)
    candidate c (exposed at record E[last position of c in line 1]) survives iff M[c] < E[..]."""
    first = bytes(st.first_name[:st.first_len]).decode('latin-1')
    last = bytes(st.last_name[:st.last_len]).decode('latin-1')
    flen = len(first)
    lcp_first = [st.first_lcp_eq[j] for j in range(flen + 1)]
    lcs_first = [st.first_lcs_eq[j] for j in range(flen + 1)]

    def running_first(arr):
        out, best = [], L.NONE_I64
        for v in arr:
            best = min(best, v)
            out.append(best)
        return out
    E = running_first(lcp_first)
    Es = running_first(lcs_first)
    # Q8: a QNAME that is a proper prefix (suffix) of the running prefix (suffix) raises IndexError
    # in the reference (uq.py:397, 405)
    for j in range(flen):
        k = st.first_short_prefix[j]
        if not _none(k) and E[j] == k:
            raise UQError('ERROR: QNAME of record %d is a proper prefix of the common QNAME prefix (the reference raises IndexError here, Q8)' % k)
        k = st.first_short_suffix[j]
        if not _none(k) and Es[j] == k:
            raise UQError('ERROR: QNAME of record %d is a proper suffix of the common QNAME suffix (the reference raises IndexError here, Q8)' % k)

    plen, slen = int(st.prefix_len), int(st.suffix_len)
    prefix = first[:plen]
    suffix = first[flen - slen:] if slen else ''
    # candidates in the reference's insertion order: by shrink event (in time order), then by position
    events = []                                    # (new, old): the running prefix shrinks from old to new
    low = sorted((lcp_first[j], j) for j in range(flen) if not _none(lcp_first[j]))    # by record index
    cur = flen
    for _, j in low:
        if j < cur:
            events.append((j, cur))                # exposes first[j:cur]
            cur = j
    sep_count = {}
    for new, old in events:
        for ch in first[new:old]:
            if ch not in sep_count:
                sep_count[ch] = None
    for ch in list(sep_count):
        k_c = E[first.rindex(ch)]
        if st.last_count_mismatch[ord(ch)] >= k_c:
            del sep_count[ch]                      # uq.py:410-413
        else:
            sep_count[ch] = first[plen:].count(ch)
    for ch in list(sep_count):                     # uq.py:428-431
        k = suffix.count(ch)
        if k:
            sep_count[ch] -= k
            if sep_count[ch] == 0:
                del sep_count[ch]
    if len(sep_count) == 0:
        raise UQError('ERROR: no QNAME separators (the reference crashes on such files, Q6)')

    def order_seps(name, cls=None):                # uq.py:433-436
        return ''.join(re.findall('([' + (cls if cls is not None else ''.join(sep_count)) + ']+)', name[len(prefix):-1 - len(suffix)]))
    try:
        a, b = order_seps(last), order_seps(first)
    except re.error as e:
        raise UQError('ERROR: QNAME separators %r break the reference regex (Q11): %s' % (''.join(sep_count), e))
    # The reference pastes the separator characters into a character class unescaped (in dict order): '-' between two
    # others silently becomes a RANGE (':-_' takes in A-Z), a leading '^' negates the class.  Such a class is only accepted
    # when it behaves like the set of characters it was meant to be; otherwise the file is refused (Q11).
    if any(ch in '-^]\\' for ch in sep_count):
        meant = ''.join(re.escape(ch) for ch in sep_count)
        if (a, b) != (order_seps(last, meant), order_seps(first, meant)):
            raise UQError('ERROR: QNAME separators %r change meaning inside the reference regex class (Q11)' % ''.join(sep_count))
    if a != b:                                     # uq.py:438-444
        raise UQError("ERROR: Sorry, the separators used in this file's QNAME/headers are so unusual/improbable that "
                      "I didn't think it was worth the time to write the code on how to deal with it, only identify it.")
    return prefix, suffix, a


def bits_for(n, pad):
    """uq.py:497-503 / uq.py:534-540."""
    if n <= 4: return 2
    if n <= 8 and not pad: return 3
    if n <= 16: return 4
    if n <= 32 and not pad: return 5
    if n <= 64 and not pad: return 6
    if n <= 128 and not pad: return 7
    return 8


def decide_alphabets(st, notricks=False, pad=False):
    base_graph = {chr(i): int(st.base_count[i]) for i in range(256) if st.base_count[i]}
    qual_graph = {chr(i): int(st.qual_count[i]) for i in range(256) if st.qual_count[i]}
    bases = sorted(base_graph)                     # uq.py:456-457
    quals = sorted(qual_graph)
    n_qual = {}
    n_qual_symbol = {}
    total_quals = len(quals)
    if not notricks:                               # uq.py:479-494
        for base in sorted(base_graph):            # py2 dict order in the reference; only matters for >=2 tricked bases (Q10)
            if len(bases) == 1:
                continue
            single = st.base_single_qual[ord(base)]
            if 0 <= single <= 255:
                bases.remove(base)
                q = chr(single)
                if base_graph[base] == qual_graph[q]:
                    n_qual[base] = quals.index(q)
                else:
                    total_quals += 1
                    n_qual[base] = total_quals     # Q3: a code with no entry in `qualities`
                    n_qual_symbol[base] = q        # the quality character that code stands for (see config_of)
    bpb = bits_for(len(bases), pad)
    dna_max = int(st.dna_max)
    variable = int(st.dna_min) != dna_max
    bpq = bits_for(total_quals, pad)
    return dict(bases=''.join(bases), qualities=''.join(quals), N_qual=n_qual, N_qual_symbol=n_qual_symbol, bits_per_base=bpb,
                bits_per_quality=bpq, variable_read_lengths=variable, dna_max=dna_max,
                dna_bytes=-(-(bpb * (dna_max + variable)) // 8), qual_bytes=-(-(bpq * (dna_max + variable)) // 8),
                base_distribution=base_graph, qual_distribution=qual_graph)


def pack_params(dec):
    p = L.PackParams()
    for i, ch in enumerate(dec['bases']):
        p.base_code[ord(ch)] = i
    for i, ch in enumerate(dec['qualities']):
        p.qual_code[ord(ch)] = i
    for i in range(256):
        p.trick_qual[i] = -1
    for base, code in dec['N_qual'].items():
        if code >> dec['bits_per_quality']:
            raise UQError('ERROR: the N-trick quality code %d does not fit %d bits; the reference corrupts its output here (Q4)'
                          % (code, dec['bits_per_quality']))
        p.trick_qual[ord(base)] = code
    p.bits_per_base, p.bits_per_quality = dec['bits_per_base'], dec['bits_per_quality']
    p.dna_bytes, p.qual_bytes = dec['dna_bytes'], dec['qual_bytes']
    p.variable, p.dna_max = int(dec['variable_read_lengths']), dec['dna_max']
    return p


# ------------------------------------------------------------------------------------------------
# Pass-2 decisions (uq.py:586-602, 641-676)
# ------------------------------------------------------------------------------------------------
def decide_columns(colstats, n_reads, fetch_dict, exact_ints=False):
    """exact_ints (the single QNAME column of E2): a column counts as all-integer only when every token is the
    canonical text of an int64 (str(int(t)) == t), so that integers decode to exactly the names they came from."""
    columns = []
    last = n_reads - 1
    for i, cs in enumerate(colstats):
        col = {'name': 'QNAME_%d' % (i + 1)}
        all_int = cs.all_int
        if exact_ints:
            all_int = cs.all_int and cs.all_canonical and not cs.overflow
        elif cs.overflow:
            raise UQError('ERROR: QNAME column %d holds an integer outside the int64 range' % (i + 1))
        demoted = False
        t = 10000
        for k in range(cs.n_checkpoints):          # uq.py:634-636
            if cs.distinct_at[k] > t // 10:
                demoted = True
                break
            t *= 2
        if not demoted and cs.n_distinct > last // 10:       # uq.py:638
            demoted = True
        if demoted:
            if not all_int:                        # 'strings' (uq.py:598-601, 624-630); the reference stops at uq.py:672-673
                # declared extension E1: the tokens themselves, zero padded to the longest one over ALL records (the
                # reference's own `longest` undercounts after an integers -> strings switch).  An all-empty column still
                # gets one byte: numpy has no zero-width S dtype.
                w = int(cs.max_len)
                if w > STRING_MAX:
                    raise UQError('ERROR: QNAME column %d holds a token of %d bytes; a string column holds at most %d'
                                  % (i + 1, w, STRING_MAX))
                col['format'] = 'strings'
                col['longest'] = w
                col['dtype'] = '|S%d' % max(w, 1)
                columns.append(col)
                continue
            col['format'] = 'integers'
            col['min'], col['max'] = int(cs.min_val), int(cs.max_val)
            span = col['max'] - col['min']
            cap, col['dtype'], _ = next(d for d in _DT if span <= d[0])
            col['offset'] = bool(col['min'] < 0 or col['max'] > cap)
        else:
            n = int(cs.n_distinct)
            cap, col['dtype'], _ = next(d for d in _DT if n <= d[0])
            if all_int and int(cs.max_val) - int(cs.min_val) <= cap:        # uq.py:649-658
                col['format'] = 'integers'
                col['max'], col['min'] = int(cs.max_val), int(cs.min_val)
                col['offset'] = bool(col['min'] < 0 or col['max'] > cap)
            else:
                col['format'] = 'mapping'
                col['map'] = fetch_dict(i)         # sorted distinct tokens (uq.py:659-661)
        if col['format'] == 'integers' and not col['offset'] and col['min'] < 0:
            raise UQError('ERROR: negative integers in QNAME column %d' % (i + 1))
        columns.append(col)
    return columns


def decide_qname_columns(st, n_reads, scan, shortest_remainder, fetch_dict):
    """QNAME layout and column typing -> (prefix, suffix, separators, columns).

    scan(prefix, suffix, separators) -> (column statistics, bad_record) tokenises every record;
    shortest_remainder(prefix_len) -> min over all records of len(name) - prefix_len.

    A file whose names the reference cuts into columns (derive_qname_layout accepts it and every record holds the
    separators in their order) gets exactly the reference's layout.  Every other file takes declared extension E2
    (DESIGN section 4): no separators and one column QNAME_1, the part of each name between the longest common prefix
    of all names and the longest common suffix of what that prefix leaves of them.  That suffix is the common suffix
    of the names clamped to the shortest remainder: unclamped, it could overlap the prefix inside a short name
    ('@ab' / '@abab'), whose middle the tokeniser would then cut empty."""
    try:
        prefix, suffix, separators = derive_qname_layout(st, n_reads)
    except UQError:
        pass
    else:
        colstats, bad = scan(prefix, suffix, separators)
        if bad < 0:
            return prefix, suffix, separators, decide_columns(colstats, n_reads, fetch_dict)
    first = bytes(st.first_name[:st.first_len]).decode('latin-1')
    plen = int(st.prefix_len)
    slen = min(int(st.suffix_len), shortest_remainder(plen))
    prefix, suffix = first[:plen], first[len(first) - slen:] if slen else ''
    colstats, bad = scan(prefix, suffix, '')
    if bad >= 0:                                   # with no separator every record is one column
        raise UQError('ERROR: record %d does not split into one QNAME column' % bad)
    return prefix, suffix, '', decide_columns(colstats, n_reads, fetch_dict, exact_ints=True)


def column_specs(columns):
    out = []
    for c in columns:
        size = np.dtype(c['dtype']).itemsize
        if c['format'] == 'mapping':
            out.append((0, size, False, 0))
        elif c['format'] == 'strings':
            out.append((2, size, False, 0))
        else:
            out.append((1, size, c['offset'], c['min'] if c['offset'] else 0))
    return out


# ------------------------------------------------------------------------------------------------
# run_mix on the device (uq.py:739-851)
# ------------------------------------------------------------------------------------------------
def key_itemsize(n_unique):
    """numpy.min_scalar_type(max(key)) with max(key) = n_unique - 1 (uq.py:790, 832)."""
    m = max(n_unique - 1, 0)
    return next(d[2] for d in _DT if m <= d[0])


class DeviceMembers:
    """Output members kept in HBM: name -> (DeviceArray, kind, meta).  download() turns them into the
    exact ndarray objects the reference hands to numpy.save.

    With a `sink` (callable (name, nbytes) -> uint8 ndarray over pinned host memory) every member starts
    its device->host copy on the copy stream the moment it is final, so the copies overlap the rest of
    the encode; download() then only waits for the copy stream."""

    def __init__(self, ctx=None, sink=None):
        self.items = {}
        self.ctx, self.sink, self.host = ctx, sink, {}
        self.order = None       # run_mix: uint32 DeviceArray, container row -> input record (None: rows in input order)

    def _queue(self, name, arr):
        if self.sink is not None:
            buf = self.sink(name, arr.nbytes)
            arr.download_async(buf)
            self.host[name] = buf

    def add_table(self, name, stream, n, width, pattern):
        self.items[name] = (stream, 'table', (n, width, pattern))
        self._queue(name, stream)

    def add_vector(self, name, arr, dtype):
        self.items[name] = (arr, 'vector', np.dtype(dtype))
        self._queue(name, arr)

    def nbytes(self):
        return sum(a.nbytes for a, _, _ in self.items.values())

    def download(self, into=None):
        out = {}
        if self.sink is not None:
            self.ctx.copy_sync()
        for name, (arr, kind, meta) in self.items.items():
            if self.sink is not None:
                flat = self.host[name][:arr.nbytes]
            else:
                buf = None if into is None else into(name, arr.nbytes)
                flat = arr.download(dtype=np.uint8, out=buf).reshape(-1)
            if kind == 'vector':
                out[name] = flat.view(meta).reshape(-1)
            else:
                n, width, pattern = meta
                out[name] = table_ndarray(flat, n, width, pattern)
        return out

    def free(self):
        if self.sink is not None and self.ctx is not None:
            self.ctx.copy_sync()
        for a, _, _ in self.items.values():
            a.free()
        self.items = {}
        if self.order is not None:
            self.order.free()
            self.order = None

    def __del__(self):
        # members dropped without free() (an exception in the middle of run_mix): the queued device->host copies must
        # finish before the garbage-collected arrays are recycled by the arena
        try:
            if self.items and self.sink is not None and self.ctx is not None and self.ctx.h:
                self.ctx.copy_sync()
        except Exception:
            pass


def table_ndarray(flat, n, width, pattern):
    """stream bytes of a laid-out table -> the ndarray object the reference hands to numpy.save (shape and memory
    order of uq.py:263-270): (N, B) for patterns 0.x / 2.x, (B, N) for 1.x / 3.x; C order for x.1, Fortran for x.2"""
    shape = (n, width) if pattern[0] in '02' else (width, n)
    return np.ndarray(shape, dtype=np.uint8, buffer=flat, order='C' if pattern[2] == '1' else 'F')


def stream_of(arr):
    """ndarray as numpy.load returns a DNA / QUAL member -> its byte stream (memory order), no copy"""
    if arr.flags.c_contiguous:
        return arr.reshape(-1)
    if arr.flags.f_contiguous:
        return arr.T.reshape(-1)
    return np.ascontiguousarray(arr).reshape(-1)


def stream_rows(arr, pattern, a, b):
    """The part of a laid-out member that holds the logical rows [a, b): contiguous uint8 bytes which are exactly the
    stream of those rows alone under the same pattern (so uqb_unlayout on them yields rows a..b-1 in order).  Row-major
    streams: one byte range (from the other end when the pattern reverses the rows); column-major streams: one run per
    byte column.  This is how a rank of the sharded decode picks its share of a member."""
    n, width = arr.shape if pattern[0] in '02' else arr.shape[::-1]
    transposed, rev_r, _ = PATTERN_DESC[pattern]
    flat = stream_of(arr)
    first = n - b if rev_r else a
    if not transposed:
        return np.ascontiguousarray(flat[first * width:(first + b - a) * width])
    return np.ascontiguousarray(flat.reshape(width, n)[:, first:first + b - a]).reshape(-1)


def _layout(ctx, table, pattern):
    """-> (stream DeviceArray, aliased).  Pattern 0.1 IS the table's own byte order: no kernel, no copy."""
    if pattern == '0.1':
        return table, True
    return ctx.layout(table, pattern), False


def _keyed(ctx, table, order):
    """numpy.unique(return_inverse) + the ordering of the key (uq.py:786-798 / 830-836).
    -> (key in output order as uint32 DeviceArray, uniq, n_unique, order)"""
    if order is False:
        # this table defines the order: key[argsort(key)] is the group id in sorted order
        perm, _, uniq, nu, key = ctx.sort_rows(table, want_perm=True, want_uniq=True, want_key_sorted=True)
        return key, uniq, nu, perm
    _, key, uniq, nu = ctx.sort_rows(table, want_key=True, want_uniq=True)
    if order is not None:
        k2 = ctx.gather_rows(key, order)
        key.free()
        key = k2
    return key, uniq, nu, order


def _prepare_keyed(ctx, out, table, name, pattern):
    """Order-independent half of a keyed DNA/QUAL table that does not define the sort order: unique table
    (emitted at once, so that its device->host copy can start) and the row -> unique-index key."""
    _, key, uniq, nu = ctx.sort_rows(table, want_key=True, want_uniq=True)         # uq.py:786
    stream, aliased = _layout(ctx, uniq, pattern)
    out.add_table(name, stream, uniq.n, uniq.width, pattern)
    if not aliased:
        uniq.free()
    return key, nu


def _mix_dna_qual(ctx, out, table, name, order, raw, pattern, prepared=None):
    """encode_dna_qual (uq.py:765-805).  order: None / False / DeviceArray(uint32 perm)."""
    if raw:
        src = table
        if order is not None:
            if order is False:
                order, _, _, _ = ctx.sort_rows(table, want_perm=True)              # uq.py:775
            src = ctx.gather_rows(table, order)                                    # uq.py:777
        stream, aliased = _layout(ctx, src, pattern)
        out.add_table(name + '.raw', stream, table.n, table.width, pattern)
        if src is not table and not aliased:
            src.free()
    elif prepared is not None:
        key, nu = prepared
        if order is not None:
            k2 = ctx.gather_rows(key, order)                                       # key[sort_order], uq.py:798
            key.free()
            key = k2
        out.add_vector(name + '.key', *_narrow_key(ctx, key, nu))                  # uq.py:790
    else:
        key, uniq, nu, order = _keyed(ctx, table, order)                           # uq.py:786, 796
        out.add_vector(name + '.key', *_narrow_key(ctx, key, nu))                  # uq.py:790
        stream, aliased = _layout(ctx, uniq, pattern)
        out.add_table(name, stream, uniq.n, uniq.width, pattern)
        if not aliased:
            uniq.free()
    return order


def qname_kinds(columns):
    """per column: 1 = 'strings' (its bytes go into the sort row as they are, E1), 0 = integer value (big-endian in the
    row); None when every column is an integer column"""
    kinds = [1 if c['format'] == 'strings' else 0 for c in columns]
    return kinds if any(kinds) else None


def qname_rows(ctx, cols, columns):
    """QNAME columns -> sort rows, whose memcmp order is the row order of E1: column by column, integers and mapping
    ranks as unsigned numbers (uq.py:814-816, 828-830), strings bytewise like numpy compares S values"""
    return ctx.columns_to_rows(cols, qname_kinds(columns))


def qname_key_plan(columns):
    """One packed 64-bit sort key for QNAME columns -> [(shift, bits, base)] per column, or None (a 'strings' column, or
    more than 64 bits).  Field c holds the column's encoded value minus `base` in `bits` bits at `shift`, the first
    column in the highest bits, so the key's numeric order is the memcmp order of qname_rows: sorting the key alone
    sorts the table, and the unique keys unpack straight into the columns."""
    fields = []
    for c in columns:
        if c['format'] == 'strings':
            return None
        if c['format'] == 'mapping':                       # rank in the sorted dictionary
            fields.append(((len(c['map']) - 1).bit_length(), 0))
        else:                                              # an offset column already holds value - min
            fields.append(((c['max'] - c['min']).bit_length(), 0 if c['offset'] else c['min']))
    if sum(b for b, _ in fields) > 64:
        return None
    plan, shift = [], 0
    for bits, base in reversed(fields):
        plan.append((shift, bits, base))
        shift += bits
    return plan[::-1]


def qname_sort_table(ctx, cols, columns):
    """QNAME columns -> (table that uqb_sort_rows sorts into the row order of E1, plan): the packed-key table when
    qname_key_plan gives one (plan), else the sort rows (None)"""
    plan = qname_key_plan(columns)
    if plan is None:
        return qname_rows(ctx, cols, columns), None
    return ctx.columns_to_key(cols, plan), plan


def qname_columns(ctx, uniq, columns, plan):
    """unique rows of the qname_sort_table table -> typed QNAME columns again (uq.py:842-847)"""
    sizes = [np.dtype(m['dtype']).itemsize for m in columns]
    if plan is None:
        return ctx.rows_to_columns(uniq, sizes, qname_kinds(columns))
    return ctx.key_to_columns(uniq, sizes, plan)


def _narrow_key(ctx, key, nu):
    """key.astype(min_scalar_type(max(key))) (uq.py:790, 832) -> (array, dtype).  Takes over `key`: a key of four-byte
    items is that array already."""
    size = key_itemsize(nu)
    if size != 4:
        narrow = ctx.narrow_u32(key, size)
        key.free()
        key = narrow
    return key, 'uint%d' % (8 * size)


def _mix_qname(ctx, out, cols, columns, order, raw):
    """encode_qname (uq.py:808-851)."""
    if raw:
        if order is False:
            table, _ = qname_sort_table(ctx, cols, columns)
            order, _, _, _ = ctx.sort_rows(table, want_perm=True)                  # uq.py:816
            table.free()
        for c, meta in zip(cols, columns):
            if order is not None:
                out.add_vector(meta['name'] + '.raw', ctx.gather_rows(c, order), meta['dtype'])
            else:
                out.add_vector(meta['name'] + '.raw', c, meta['dtype'])
    else:
        table, plan = qname_sort_table(ctx, cols, columns)
        key, uniq, nu, order = _keyed(ctx, table, order)                           # uq.py:830, 833
        table.free()
        out.add_vector('QNAME.key', *_narrow_key(ctx, key, nu))
        ucols = qname_columns(ctx, uniq, columns, plan)                            # uq.py:842-847
        uniq.free()
        for c, meta in zip(ucols, columns):
            out.add_vector(meta['name'], c, meta['dtype'])
    return order


def run_mix(ctx, dna, qual, cols, columns, sorted_on, raw_tables, pattern, sink=None):
    """uq.py:739-753.  The reference runs the sorted-on table first; here the order-independent half of the
    other keyed table (its unique table - the largest output) is produced before that, so that its
    device->host copy overlaps the remaining sorts.  The results are identical.  The sort order (the stable argsort that
    links container row i to input record order[i]) stays on the members as `order` for verify_device."""
    out = DeviceMembers(ctx, sink)
    pd, pq = pattern
    if sorted_on in ('DNA', 'QUAL'):
        first = (dna, 'DNA', pd) if sorted_on == 'DNA' else (qual, 'QUAL', pq)
        second = (qual, 'QUAL', pq) if sorted_on == 'DNA' else (dna, 'DNA', pd)
        prepared = None
        if second[1] not in raw_tables:
            prepared = _timed(ctx, 'mix_' + second[1], _prepare_keyed, ctx, out, second[0], second[1], second[2])
        out.order = _timed(ctx, 'mix_' + first[1], _mix_dna_qual, ctx, out, first[0], first[1], False, first[1] in raw_tables, first[2])
        _timed(ctx, 'mix_' + second[1], _mix_dna_qual, ctx, out, second[0], second[1], out.order, second[1] in raw_tables, second[2], prepared)
        _timed(ctx, 'mix_QNAME', _mix_qname, ctx, out, cols, columns, out.order, 'QNAME' in raw_tables)
    elif sorted_on == 'QNAME':
        out.order = _timed(ctx, 'mix_QNAME', _mix_qname, ctx, out, cols, columns, False, 'QNAME' in raw_tables)
        _timed(ctx, 'mix_QUAL', _mix_dna_qual, ctx, out, qual, 'QUAL', out.order, 'QUAL' in raw_tables, pq)
        _timed(ctx, 'mix_DNA', _mix_dna_qual, ctx, out, dna, 'DNA', out.order, 'DNA' in raw_tables, pd)
    else:
        _timed(ctx, 'mix_QUAL', _mix_dna_qual, ctx, out, qual, 'QUAL', None, 'QUAL' in raw_tables, pq)
        _timed(ctx, 'mix_DNA', _mix_dna_qual, ctx, out, dna, 'DNA', None, 'DNA' in raw_tables, pd)
        _timed(ctx, 'mix_QNAME', _mix_qname, ctx, out, cols, columns, None, 'QNAME' in raw_tables)
    return out


# ------------------------------------------------------------------------------------------------
# encode
# ------------------------------------------------------------------------------------------------
def config_of(dec, n, prefix, suffix, separators, columns, sort, raw, pattern):
    """config.json (uq.py:681-696, 898-903).

    One key is added when - and only when - the N-trick took its "new quality" branch (uq.py:489-494, SURVEY Q3): the
    reference then stores a quality code that has no entry in `qualities`, its own decoder raises IndexError on such
    a file and the original quality character is written nowhere.  `N_qual_symbol` = {base: that character} makes
    the container decodable (decode_device reads it); every array and every other key stay exactly the reference's."""
    config = {
        'base_distribution': dec['base_distribution'], 'qual_distribution': dec['qual_distribution'],
        'reads': n, 'bases': dec['bases'], 'qualities': dec['qualities'],
        'variable_read_lengths': dec['variable_read_lengths'], 'bits_per_base': dec['bits_per_base'],
        'bits_per_quality': dec['bits_per_quality'], 'N_qual': dec['N_qual'], 'dna_max': dec['dna_max'],
        'QNAME_prefix': prefix, 'QNAME_suffix': suffix, 'QNAME_separators': separators,
        'QNAME_columns': columns, 'sort': sort, 'raw': list(raw), 'pattern': pattern,
    }
    if dec.get('N_qual_symbol'):
        config['N_qual_symbol'] = dict(dec['N_qual_symbol'])
    return config


def prepare(ctx, fq, pad=False, notricks=False):
    """Pass 1 - Pass 4 of the reference (uq.py:338-735) on a FASTQ that is resident in HBM: statistics, decisions,
    packed DNA / QUAL tables and encoded QNAME columns.  -> dict(stats, dec, columns, prefix, suffix, separators,
    total, dna, qual, cols); everything a mix (run_mix) or the --test feed (MixFeed) needs."""
    info = _timed(ctx, 'split', fq.split)
    if info.status == 1:                                                           # uq.py:86-87
        raise UQError('ERROR: The FASTQ file provided contains' + str(info.n_lines) + 'rows, which is not divisible by 4!')
    n = int(info.n_reads)
    if n == 0:
        raise UQError('ERROR: the FASTQ file holds no records')
    st = _timed(ctx, 'analyze', fq.analyze)
    if st.bad_first_char != -1:                                                    # uq.py:346
        raise UQError('ERROR: This does not look like a FASTA/FASTQ file! (first line does not start with @)')
    bad = [(r, w) for r, w in ((st.bad_plus_record, 'plus'), (st.bad_len_record, 'len')) if r >= 0]
    if bad:
        r, w = min(bad, key=lambda t: (t[0], t[1] != 'plus'))
        if w == 'plus':                                                            # uq.py:360, 382
            raise UQError('ERROR: For entry %d the third line does not start with +' % r)
        raise UQError('ERROR: Length of DNA does not match the length of the quality scores for entry %d' % (r + 1))   # uq.py:366, 388
    prefix, suffix, separators, columns = decide_qname_columns(
        st, n, lambda p, s, seps: _timed(ctx, 'qname_scan', fq.qname_scan, len(p), len(s), seps),
        lambda plen: int(_timed(ctx, 'qname_remainder', fq.qname_scan, plen, 0, '', col_mode=[1])[0][0].min_len),
        fq.qname_dict)
    dec = decide_alphabets(st, notricks=notricks, pad=pad)
    dna, qual = _timed(ctx, 'pack', fq.pack, pack_params(dec))
    cols = _timed(ctx, 'qname_encode', fq.qname_encode, column_specs(columns))
    return dict(stats=st, dec=dec, columns=columns, dna=dna, qual=qual, cols=cols, prefix=prefix, suffix=suffix,
                separators=separators, total=n)


def encode_device(ctx, fq, sort=None, raw=None, pattern=None, pad=False, notricks=False, stages=None, sink=None):
    """FASTQ already in HBM (device.Fastq) -> (DeviceMembers, config).  All O(N) work is on the GPU."""
    sort, raw, pattern = normalise_options(sort, raw, pattern)
    p = prepare(ctx, fq, pad=pad, notricks=notricks)
    dna, qual, cols, columns = p['dna'], p['qual'], p['cols'], p['columns']
    if stages is not None:
        stages.update(p)
    members = run_mix(ctx, dna, qual, cols, columns, sort, raw, pattern, sink=sink)
    if stages is None:
        keep = {id(a) for a, _, _ in members.items.values()}
        for a in [dna, qual] + cols:
            if id(a) not in keep:
                a.free()
    return members, config_of(p['dec'], p['total'], p['prefix'], p['suffix'], p['separators'], columns, sort, raw, pattern)


class MixFeed:
    """Device-resident feed of the --test search (test_patterns uq.py:290-334, loop uq.py:855-889; SURVEY section 8 f1).

    The reference re-sorts, re-uniques and rot90s its tables for every candidate mix.  Here the FASTQ is loaded and
    Pass 1-4 run ONCE; the packed tables stay in HBM, each of DNA / QUAL / QNAME is sorted at most once (one
    uqb_sort_rows gives its stable argsort, its unique table and its key both in record and in sorted order), and a
    member of any (sort, raw, pattern) mix is then only a gather (uqb_gather_rows) and / or a layout (uqb_layout) of
    cached arrays.  members(sort, raw, pattern) returns host ndarrays exactly like encode() - same bytes, same dtypes,
    same memory order - so the compressor / argmin side of --test stays the reference's."""

    def __init__(self, ctx, fq, pad=False, notricks=False):
        self.ctx = ctx
        self.p = prepare(ctx, fq, pad=pad, notricks=notricks)
        self.tables = {'DNA': self.p['dna'], 'QUAL': self.p['qual'], 'QNAME': None}
        self.qname_plan = None
        self.sorted = {}            # table -> dict(perm, key, key_sorted, uniq, nu)
        self.cache = {}             # derived device arrays: ('rows', T, S) / ('key', T, S) / ('stream', ...) ...
        self.kernel_launches_after_prepare = ctx.launches

    def config(self, sort, raw, pattern):
        sort, raw, pattern = normalise_options(sort, raw, pattern)
        p = self.p
        return config_of(p['dec'], p['total'], p['prefix'], p['suffix'], p['separators'], p['columns'], sort, raw, pattern)

    def _table(self, t):
        if self.tables[t] is None:                       # QNAME sort rows (uq.py:814-816)
            self.tables[t], self.qname_plan = qname_sort_table(self.ctx, self.p['cols'], self.p['columns'])
        return self.tables[t]

    def _sorted(self, t):
        if t not in self.sorted:
            perm, key, uniq, nu, key_sorted = self.ctx.sort_rows(self._table(t), want_perm=True, want_key=True, want_uniq=True,
                                                                 want_key_sorted=True)
            self.sorted[t] = dict(perm=perm, key=key, uniq=uniq, nu=nu, key_sorted=key_sorted)
        return self.sorted[t]

    def _cached(self, tag, make):
        if tag not in self.cache:
            self.cache[tag] = make()
        return self.cache[tag]

    def _host_table(self, tag, rows, pattern):
        """laid-out table -> ndarray as handed to numpy.save; the stream is produced on the device once per (table, pattern)"""
        def make():
            if pattern == '0.1':
                return rows.download(dtype=np.uint8).reshape(-1)
            stream = self.ctx.layout(rows, pattern)
            flat = stream.download(dtype=np.uint8).reshape(-1)
            stream.free()
            return flat
        flat = self._cached(('stream',) + tag + (pattern,), make)
        return table_ndarray(flat, rows.n, rows.width, pattern)

    def members(self, sort=None, raw=None, pattern=None):
        ctx = self.ctx
        sort, raw, pattern = normalise_options(sort, raw, pattern)
        s_on = sort if sort in ('DNA', 'QUAL', 'QNAME') else None
        order = self._sorted(s_on)['perm'] if s_on else None                         # uq.py:775, 796, 816, 833
        out = {}
        for t, pat in (('DNA', pattern[0]), ('QUAL', pattern[1])):
            if t in raw:                                                             # uq.py:767-781
                rows = self.tables[t] if order is None else self._cached(('rows', t, s_on), lambda: ctx.gather_rows(self.tables[t], order))
                out[t + '.raw'] = self._host_table(('raw', t, s_on), rows, pat)
            else:                                                                    # uq.py:783-802
                srt = self._sorted(t)
                out[t + '.key'] = self._key(t, s_on, order)
                out[t] = self._host_table(('uniq', t), srt['uniq'], pat)
        columns = self.p['columns']
        if 'QNAME' in raw:                                                           # uq.py:812-826
            for c, meta in zip(self.p['cols'], columns):
                def make(c=c):
                    if order is None:
                        return c.download(dtype=np.dtype(meta['dtype'])).reshape(-1)
                    g = ctx.gather_rows(c, order)
                    h = g.download(dtype=np.dtype(meta['dtype'])).reshape(-1)
                    g.free()
                    return h
                out[meta['name'] + '.raw'] = self._cached(('qcol', meta['name'], s_on), make)
        else:                                                                        # uq.py:827-847
            srt = self._sorted('QNAME')
            out['QNAME.key'] = self._key('QNAME', s_on, order)

            def make_cols():
                ucols = qname_columns(ctx, srt['uniq'], columns, self.qname_plan)
                host = [u.download(dtype=np.dtype(m['dtype'])).reshape(-1) for u, m in zip(ucols, columns)]
                for u in ucols:
                    u.free()
                return host
            for h, meta in zip(self._cached(('qucols',), make_cols), columns):
                out[meta['name']] = h
        return out

    def _key(self, t, s_on, order):
        """key of table t in the order of the mix, narrowed like key.astype(min_scalar_type(max(key))) (uq.py:790, 832)"""
        def make():
            srt = self._sorted(t)
            size = key_itemsize(srt['nu'])
            if t == s_on:
                k32, tmp = srt['key_sorted'], None                                   # key[argsort(key)]
            elif order is None:
                k32, tmp = srt['key'], None
            else:
                k32 = tmp = self.ctx.gather_rows(srt['key'], order)                  # key[sort_order], uq.py:798
            narrow = k32 if size == 4 else self.ctx.narrow_u32(k32, size)
            h = narrow.download(dtype=np.dtype('uint%d' % (8 * size))).reshape(-1)
            if narrow is not k32:
                narrow.free()
            if tmp is not None:
                tmp.free()
            return h
        return self._cached(('key', t, s_on), make)

    def free(self):
        for d in self.sorted.values():
            for k in ('perm', 'key', 'uniq', 'key_sorted'):
                d[k].free()
        for tag, v in self.cache.items():
            if isinstance(v, DeviceArray):
                v.free()
        if self.tables['QNAME'] is not None:
            self.tables['QNAME'].free()
        for a in [self.p['dna'], self.p['qual']] + self.p['cols']:
            a.free()
        self.sorted, self.cache = {}, {}


def encode(fastq, sort=None, raw=None, pattern=None, pad=False, notricks=False, ctx=None, stages=None):
    """FASTQ bytes on the host -> (members: name -> ndarray as handed to numpy.save, config)."""
    own = ctx is None
    ctx = ctx or Context()
    fq = ctx.load_fastq(fastq)
    try:
        members, config = encode_device(ctx, fq, sort, raw, pattern, pad, notricks, stages)
        host = members.download()
        if stages is None:
            members.free()
        else:
            stages['device_members'] = members
        return host, config
    finally:
        fq.free()
        if own and stages is None:
            ctx.close()


# ------------------------------------------------------------------------------------------------
# decode (uq.py:939-1058)
# ------------------------------------------------------------------------------------------------
def _upload_table(ctx, members, name, pattern):
    """DNA / QUAL member(s) -> logical DeviceArray [n][width] (load_from_tar + key expansion)."""
    def logical(arr):
        n, width = arr.shape if pattern[0] in '02' else arr.shape[::-1]
        flat = np.ascontiguousarray(arr.ravel(order='K') if (arr.flags.c_contiguous or arr.flags.f_contiguous) else arr.ravel())
        # numpy.load returns fortran_order arrays F-contiguous: ravel('K') is the file's byte stream
        stream = ctx.upload(flat, width=1)
        tab = ctx.unlayout(stream, n, width, pattern)                              # uq.py:943-945
        stream.free()
        return tab
    if name + '.raw' in members:
        return logical(members[name + '.raw'])
    if name in members and name + '.key' in members:
        uniq = logical(members[name])
        key = _upload_key(ctx, members[name + '.key'], uniq.n, name + '.key')
        tab = ctx.gather_rows(uniq, key)                                           # uq.py:953, 957
        uniq.free(); key.free()
        return tab
    raise UQError('ERROR: No %s data was found in this uQ file?!' % name)


def _upload_key(ctx, key, n_rows, name):
    """index member in its own dtype -> uint32 DeviceArray; every value must index the table it belongs to (a malformed
    container must fail here, not fault in the gather: the reference raises IndexError at uq.py:953/957/973)."""
    key = np.ascontiguousarray(key)
    if key.dtype.kind not in 'ui' or key.ndim != 1:
        raise UQError('ERROR: %s is not a one-dimensional integer array' % name)
    if key.dtype.kind == 'i':
        if key.size and int(key.min()) < 0:
            raise UQError('ERROR: %s holds a negative index' % name)
        key = key.view(np.dtype('uint%d' % (8 * key.dtype.itemsize)))
    raw = ctx.upload(key)
    k32, bad = ctx.index_u32(raw, n_rows)
    raw.free()
    if bad >= 0:
        k32.free()
        raise UQError('ERROR: %s[%d] points outside its table of %d rows (malformed uQ file)' % (name, bad, n_rows))
    return k32


def decode_device(ctx, dna, qual, dcols, config):
    """Logical tables already in HBM (dna / qual: [n][bytes]; dcols: one DeviceArray per QNAME column,
    already expanded through QNAME.key) -> DeviceArray holding the FASTQ text (uq.py:1002-1058)."""
    import ctypes as C
    cols_meta = config['QNAME_columns']
    ncol = len(cols_meta)
    p = L.DecodeParams()
    for i, ch in enumerate(config['bases']):
        p.base_char[i] = ord(ch)
    for i, ch in enumerate(config['qualities']):
        p.qual_char[i] = ord(ch)
    for i in range(256):
        p.qual_to_base[i] = -1
    for base, code in config['N_qual'].items():                                    # qual_N, uq.py:999
        if not 0 <= code <= 255:
            raise UQError('ERROR: N_qual code %r is out of range' % (code,))
        if code >= len(config['qualities']):
            # "new quality" branch of the N-trick (Q3): the code has no entry in `qualities`
            sym = config.get('N_qual_symbol', {}).get(base)
            if sym is None:
                raise UQError('ERROR: N_qual code %d has no quality symbol; the reference decoder raises IndexError here (Q3)' % code)
            p.qual_char[code] = ord(sym)
        p.qual_to_base[code] = ord(base)
    p.bits_per_base, p.bits_per_quality = config['bits_per_base'], config['bits_per_quality']
    p.variable, p.dna_max = int(config['variable_read_lengths']), config['dna_max']
    keep = []
    def cbuf(s):
        b = np.frombuffer(s.encode('latin-1'), dtype=np.uint8).copy() if s else np.zeros(1, np.uint8)
        keep.append(b)
        return b.ctypes.data_as(C.c_void_p)
    p.prefix, p.prefix_len = cbuf(config['QNAME_prefix']), len(config['QNAME_prefix'])
    p.suffix, p.suffix_len = cbuf(config['QNAME_suffix']), len(config['QNAME_suffix'])
    p.seps, p.nseps = cbuf(config['QNAME_separators']), len(config['QNAME_separators'])
    p.ncols = ncol
    carr = (L.DecodeCol * max(ncol, 1))()
    for i, meta in enumerate(cols_meta):
        carr[i].itemsize = np.dtype(meta['dtype']).itemsize
        if meta['format'] == 'mapping':
            carr[i].format = 0
            words = [w.encode('latin-1') for w in meta['map']]
            width = max([len(w) for w in words] + [1])
            d = np.zeros((max(len(words), 1), width), dtype=np.uint8)
            for k, w in enumerate(words):
                d[k, :len(w)] = np.frombuffer(w, dtype=np.uint8)
            keep.append(d)
            carr[i].dict = d.ctypes.data_as(C.c_void_p)
            carr[i].dict_count, carr[i].dict_width = len(words), width
        elif meta['format'] == 'integers':
            carr[i].format = 1
            carr[i].offset = 1 if meta['offset'] else 0
            carr[i].min_val = int(meta['min']) if meta['offset'] else 0
        elif meta['format'] == 'strings':                                          # E1 (the reference stops, uq.py:1020-1021)
            w = np.dtype(meta['dtype'])
            if w.kind != 'S' or not 1 <= w.itemsize <= STRING_MAX:
                raise UQError('ERROR: QNAME column %d: a string column needs dtype |S1 .. |S%d, not %s' % (i + 1, STRING_MAX, w.str))
            carr[i].format = 2
        else:
            raise UQError('ERROR: QNAME column %d has the unknown format %r' % (i + 1, meta['format']))
    p.cols = carr
    h = C.c_void_p()
    handles = (C.c_void_p * max(ncol, 1))(*[c.h for c in dcols])
    ctx.check(ctx.lib.uqb_decode(ctx.h, dna.h, qual.h, handles, C.byref(p), C.byref(h)))
    return DeviceArray(ctx, h)


class MemberRows:
    """The decoder's front (load_from_tar + key expansion, uq.py:943-973) on members that are already in HBM (a
    DeviceMembers as encode_device returns it), for any range of container rows [a, b): rows(a, b) -> (dna, qual, dcols),
    the logical tables and the QNAME columns of those rows, ready for decode_device.  Streams are un-laid-out, keys widened
    and bound-checked, rows gathered - all on the device.

    A raw pattern-0.1 stream and a raw QNAME column are views of their rows.  A keyed table or QNAME column is gathered
    through a view of its key's rows, so a batch needs memory for its own rows only.  A unique table, and a raw table in
    another pattern, are un-laid-out once for the whole file (here, in the constructor).  The arrays of one rows() call
    are released by release() (or close())."""

    def __init__(self, ctx, dm, config):
        self.ctx, self.it, self.config = ctx, dm.items, config
        self.n = int(config['reads'])
        self.whole, self.batch = [], []
        try:
            self.src = {name: self._logical(name) for name in ('DNA', 'QUAL')}
        except Exception:
            self.close()
            raise

    def _logical(self, name):
        """DNA / QUAL -> (logical table of the raw rows or of the unique rows, key member name or None)"""
        def unlaid(entry):
            stream, _, (n, width, p) = entry
            if p == '0.1':
                return self._hold(self.ctx.wrap(stream.device_ptr.value, n, width), self.whole)
            return self._hold(self.ctx.unlayout(stream, n, width, p), self.whole)
        if name + '.raw' in self.it:
            return unlaid(self.it[name + '.raw']), None
        return unlaid(self.it[name]), name + '.key'

    @staticmethod
    def _hold(a, into):
        into.append(a)
        return a

    def _view(self, arr, a, b):
        """rows [a, b) of a device array: a view when it starts 16-byte aligned (the decode kernels load packed rows as
        aligned 16-byte words), else a copy of the rows"""
        w = arr.width
        ptr = arr.device_ptr.value + a * w
        if a == 0 or ptr % 16 == 0:
            return self._hold(self.ctx.wrap(ptr, b - a, w), self.batch)
        out = self._hold(self.ctx.alloc(b - a, w), self.batch)
        self.ctx.copy_in(out, 0, ptr, (b - a) * w)
        return out

    def _key(self, name, n_rows, a, b):
        k32, bad = self.ctx.index_u32(self._view(self.it[name][0], a, b), n_rows)
        self._hold(k32, self.batch)
        if bad >= 0:
            raise UQError('ERROR: %s[%d] points outside its table of %d rows (malformed uQ file)' % (name, a + bad, n_rows))
        return k32

    def _rows(self, table, key, a, b):
        if key is None:
            return self._view(table, a, b)
        return self._hold(self.ctx.gather_rows(table, self._key(key, table.n, a, b)), self.batch)      # uq.py:953, 957

    def rows(self, a, b):
        self.release()
        dna, qual = (self._rows(t, k, a, b) for t, k in (self.src['DNA'], self.src['QUAL']))
        keyed = 'QNAME.key' in self.it
        dcols, key = [], None
        for meta in self.config['QNAME_columns']:
            c = self.it[meta['name'] + ('' if keyed else '.raw')][0]
            if keyed:
                if key is None:
                    key = self._key('QNAME.key', c.n, a, b)
                dcols.append(self._hold(self.ctx.gather_rows(c, key), self.batch))                     # uq.py:973
            else:
                dcols.append(self._view(c, a, b))
        return dna, qual, dcols

    def release(self):
        for x in self.batch:
            x.free()
        self.batch = []

    def close(self):
        self.release()
        for x in self.whole:
            x.free()
        self.whole = []


def decode_members_device(ctx, dm, config):
    """decode_device on members that are already in HBM (a DeviceMembers as encode_device returns it), all rows at once.
    -> DeviceArray with the FASTQ text."""
    rows = MemberRows(ctx, dm, config)
    try:
        return decode_device(ctx, *rows.rows(0, rows.n), config)
    finally:
        rows.close()


# ------------------------------------------------------------------------------------------------
# verify: the encode decoded on the device and compared with its input, record by record
# ------------------------------------------------------------------------------------------------
FIELDS = ('name', 'sequence', '+ line', 'quality')


def verify_batch_rows(ctx, fq, members, config, want=1 << 24):
    """Rows per verify batch that fit next to what is already allocated: the largest multiple of 2^20 up to `want` whose
    decoded text, line offsets and gathered rows take at most 3/4 of the device memory the context does not hold;
    0 when not even 2^20 rows fit.  (Device memory is counted as total - held: the context's arena keeps what it has
    mapped, so that is the room it can grow into.)"""
    n = int(config['reads'])
    in_use, _, total = ctx.mem_info()
    widths = 0
    once = (n + 31) // 32 * 4                                         # permutation bits
    for name, (arr, kind, meta) in members.items.items():
        if kind == 'table':
            m, width, pattern = meta
            widths += width
            if pattern != '0.1':
                once += m * width                                     # un-laid-out once for the whole file
        else:
            widths += arr.width + (4 if name.endswith('.key') else 0)
    per_row = 2 * (fq.nbytes // max(n, 1) + 1) + 4 * 8 + 12 + 2 * widths     # text (+ its copy in flight), line offsets, decode scratch
    room = (total - in_use - once) * 3 // 4
    if n <= (1 << 20):
        return n if room >= n * per_row else 0
    fit = room // per_row // (1 << 20) * (1 << 20)
    return int(min(want, fit, n)) if fit >= (1 << 20) else 0


def verify_device(ctx, fq, members, config, batch_rows=1 << 24):
    """Decode the members of an encode (a DeviceMembers from encode_device, still in HBM) batch by batch and compare
    every record with its input record in fq (the split FASTQ they were encoded from), under members.order.  Nothing is
    copied to the host but the report.
    -> dict(records, differ[4], first_row[4], first_src[4], missing, lines): per field (0 name, 1 sequence, 2 '+' line,
    3 quality) the rows whose line differs and the first such container row with its input record; `missing` the
    smallest input record that members.order does not hold (-1: a permutation, or no order); `lines[f]` = (input line,
    decoded line) of the first difference of field f, as bytes without the newline."""
    n = int(config['reads'])
    if fq.n_reads is None:
        fq.split()
    rep = L.VerifyReport()
    for f in range(4):
        rep.first_row[f] = rep.first_src[f] = -1
    order = members.order
    missing = _timed(ctx, 'verify_perm', ctx.check_permutation, order, n) if order is not None else -1
    batch_rows = max(1, int(batch_rows))
    lines = {}

    def line(h, k):
        o = h.line_offsets(k, 2)
        return h.download(int(o[0]), int(o[1] - o[0]) - 1).tobytes()

    rows = MemberRows(ctx, members, config)
    try:
        for a in range(0, n, batch_rows):
            b = min(n, a + batch_rows)
            tables = _timed(ctx, 'verify_rows', rows.rows, a, b)
            text = _timed(ctx, 'verify_decode', decode_device, ctx, *tables, config)
            rows.release()
            tfq = ctx.adopt_fastq(text)
            try:
                _timed(ctx, 'verify_split', tfq.split)
                before = list(rep.first_row)
                _timed(ctx, 'verify_compare', ctx.verify_records, fq, tfq, a, order, rep)
                for f in range(4):
                    if rep.first_row[f] >= 0 and before[f] < 0:     # the first difference of field f is in this batch
                        r, s = int(rep.first_row[f]), int(rep.first_src[f])
                        lines[f] = (line(fq, 4 * s + f) if s < fq.n_reads else None, line(tfq, 4 * (r - a) + f))
            finally:
                tfq.free()
                text.free()
    finally:
        rows.close()
    return dict(records=int(rep.records), differ=[int(x) for x in rep.differ], first_row=[int(x) for x in rep.first_row],
                first_src=[int(x) for x in rep.first_src], missing=missing, lines=lines)


def verify_clean(report):
    return not any(report['differ']) and report['missing'] < 0


def decode(members, config, ctx=None, out=None):
    """members/config as container.read_container returns them -> FASTQ bytes (uint8 ndarray).  `out`: optional
    uint8 ndarray to receive the text (e.g. over pinned memory, which makes the D2H copy run at PCIe speed)."""
    own = ctx is None
    ctx = ctx or Context()
    pat = config['pattern']
    dna = _upload_table(ctx, members, 'DNA', pat[0])
    qual = _upload_table(ctx, members, 'QUAL', pat[1])
    cols_meta = config['QNAME_columns']
    keyed = 'QNAME.key' in members
    dcols = []
    key = None
    for i, meta in enumerate(cols_meta):
        nm = 'QNAME_%d' % (i + 1) + ('' if keyed else '.raw')
        if nm not in members:
            raise UQError('ERROR: No QNAME data exists in this uQ file?')
        c = ctx.upload(np.ascontiguousarray(members[nm], dtype=meta['dtype']))
        if keyed and key is None:
            key = _upload_key(ctx, members['QNAME.key'], c.n, 'QNAME.key')
        if keyed:
            c2 = ctx.gather_rows(c, key)                                           # uq.py:973
            c.free()
            c = c2
        dcols.append(c)
    if key is not None:
        key.free()
    text = decode_device(ctx, dna, qual, dcols, config)
    if out is not None and out.size < text.nbytes:
        raise UQError('ERROR: output buffer too small (%d < %d bytes)' % (out.size, text.nbytes))
    data = text.download(out=out).reshape(-1)
    for a in [dna, qual, text] + dcols:
        a.free()
    if own:
        ctx.close()
    return data
