"""Vectorised (numpy) closed-form oracle for sizes the literal oracle cannot reach in seconds.

TEST INFRASTRUCTURE.  Implements SURVEY A.1-A.3 directly:
  * packed row = symbols concatenated most-significant first, right aligned in the row (A.1/A.2),
  * sort / unique = numpy on a void view with kind='stable' (A.3),
and is itself checked against the literal oracle (and therefore against the reference-written golden
containers) in tests/test_oracle_vec.py.  Fixed-length reads only for the packer."""
import numpy as np


def parse_fixed(fastq, read_len):
    """Fixed-length FASTQ -> (header list, dna uint8[N][L], qual uint8[N][L]) using line offsets."""
    a = np.frombuffer(fastq, dtype=np.uint8)
    nl = np.flatnonzero(a == 10)
    assert len(nl) % 4 == 0
    starts = np.concatenate([[0], nl[:-1] + 1])
    n = len(nl) // 4
    d0 = starts[1::4]
    q0 = starts[3::4]
    assert np.all(nl[1::4] - d0 == read_len) and np.all(nl[3::4] - q0 == read_len)
    idx = np.arange(read_len)
    dna = a[d0[:, None] + idx]
    qual = a[q0[:, None] + idx]
    h0, h1 = starts[0::4], nl[0::4]
    return (h0, h1), dna, qual


def pack_codes(codes, bits, width):
    """codes uint8[N][L] -> packed uint8[N][width], right-aligned big-endian bit string."""
    n, L = codes.shape
    sym_bits = ((codes[:, :, None] >> np.arange(bits - 1, -1, -1)) & 1).astype(np.uint8).reshape(n, L * bits)
    pad = width * 8 - L * bits
    full = np.zeros((n, width * 8), dtype=np.uint8)
    full[:, pad:] = sym_bits
    return np.packbits(full, axis=1)


def pack_tables(dna, qual, dec):
    """dec: the decision dict of uq_literal.decide / uq_b200.host.decide_alphabets."""
    base_code = np.zeros(256, dtype=np.uint8)
    qual_code = np.zeros(256, dtype=np.uint8)
    for i, ch in enumerate(dec['bases']): base_code[ord(ch)] = i
    for i, ch in enumerate(dec['qualities']): qual_code[ord(ch)] = i
    cd = base_code[dna]
    cq = qual_code[qual]
    for base, code in dec['N_qual'].items():
        m = dna == ord(base)
        cd[m] = 0
        cq[m] = code
    return (pack_codes(cd, dec['bits_per_base'], dec['dna_bytes']),
            pack_codes(cq, dec['bits_per_quality'], dec['qual_bytes']))


def sort_unique(table):
    v = np.ascontiguousarray(table).view('V%d' % table.shape[1]).reshape(-1)
    perm = np.argsort(v, kind='stable')
    uniq, key = np.unique(v, return_inverse=True)
    return perm, key.reshape(-1), uniq.view(np.uint8).reshape(len(uniq), table.shape[1])


def be_words(table):
    """uint8 rows -> list of big-endian 64-bit words, most significant first (the last one zero padded): comparing the
    word lists in order is memcmp order of the rows"""
    n, w = table.shape
    pad = np.zeros((n, -(-w // 8) * 8), dtype=np.uint8)
    pad[:, :w] = table
    return [pad[:, i:i + 8].copy().view('>u8').reshape(-1) for i in range(0, pad.shape[1], 8)]


def sort_unique_rows(table):
    """sort_unique through np.lexsort over big-endian words, an order of magnitude faster on millions of wide rows.
    -> (perm: stable argsort of the rows, key: unique index of every row, key_sorted = key[perm], uniq: the unique
    rows in ascending order)"""
    n, w = table.shape
    if n == 0:
        e = np.zeros(0, dtype=np.int64)
        return e, e, e, np.zeros((0, w), dtype=np.uint8)
    words = be_words(table)
    perm = np.lexsort(words[::-1])                  # stable, the first word is the primary key
    head = np.zeros(n, dtype=bool)
    head[0] = True
    for c in words:
        s = c[perm]
        head[1:] |= s[1:] != s[:-1]
    key_sorted = np.cumsum(head, dtype=np.int64) - 1
    key = np.empty(n, dtype=np.int64)
    key[perm] = key_sorted
    return perm, key, key_sorted, table[perm[head]]
