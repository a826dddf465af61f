"""Declared extension E1 (DESIGN section 4) on top of the literal oracle: 'strings' QNAME columns.

TEST INFRASTRUCTURE.  oracle/uq_literal.py restates the reference, which stops where a QNAME column leaves 'mapping'
and is not all integers (uq.py:672-673, "I havent implimented this yet").  This module is that restatement with E1 in
the four places it touches, and reuses everything else from uq_literal unchanged:

  final typing (uq.py:641-676)   a 'strings' column becomes {"format": "strings", "longest": W, "dtype": "|S<W>"},
                                 W = the longest token over ALL records (at least 1 byte, at most 255)
  Pass 4 (uq.py:717-735)         the token bytes, zero padded by numpy
  encode_qname (uq.py:808-851)   numpy.dstack cannot stack S and unsigned columns: rows are ordered with numpy.lexsort
                                 over the columns (stable, first column primary; integers as unsigned, strings as
                                 numpy compares S values); files without string columns take uq_literal's own path
  decode (uq.py:1010-1024)       a string column's text is its bytes up to the first NUL

On a file without string columns every function here returns exactly what uq_literal returns.
"""
import bisect

import numpy

from . import uq_literal as lit
from .uq_literal import UQError

STRING_MAX = 255


def pass2(lines, total, prefix, suffix, separators):
    """uq_literal.pass2 (uq.py:555-676) with E1 in the final typing"""
    ncols = None
    target = 10000
    columns = []
    last = -1
    longest = []                                            # longest token of every column over all records
    for last, toks in enumerate(lit.qname_tokens(lines, total, prefix, suffix, separators)):
        if ncols is None:                                   # uq.py:605-608
            ncols = len(toks)
            columns = [{'name': 'QNAME_%d' % (i + 1), 'format': 'mapping', 'map': set()} for i in range(ncols)]
            longest = [0] * ncols
        elif len(toks) != ncols:                            # uq.py:609-613, 637
            raise UQError('Encoding QNAMEs as strings has not been implimented yet.')
        for i, tok in enumerate(toks):                      # uq.py:614-633
            col = columns[i]
            if len(tok) > longest[i]:
                longest[i] = len(tok)
            if col['format'] == 'mapping':
                col['map'].add(tok)
            elif col['format'] == 'integers':
                try:
                    v = int(tok)
                    if v < col['min']: col['min'] = v
                    elif v > col['max']: col['max'] = v
                except ValueError:
                    col['format'] = 'strings'
                    col['longest'] = len(str(col['max']))   # the reference's own count (it can undercount)
                    del col['min'], col['max']
            elif col['format'] == 'strings':
                if len(tok) > col['longest']: col['longest'] = len(tok)
        if last == target:                                  # uq.py:634-636
            lit._demote(columns, last)
            target *= 2
    lit._demote(columns, last)                              # uq.py:638

    for i, col in enumerate(columns):                       # uq.py:641-673
        if col['format'] == 'mapping':
            n = len(col['map'])
            cap, col['dtype'] = next((m, d) for m, d in lit._DT_MAX if n <= m)
            try:
                vals = list(map(int, col['map']))
                if max(vals) - min(vals) <= cap:
                    col['format'] = 'integers'
                    col['max'], col['min'] = max(vals), min(vals)
                    col['offset'] = bool(min(vals) < 0 or max(vals) > cap)
                    del col['map']
                else:
                    col['map'] = sorted(col['map'])
            except Exception:
                col['map'] = sorted(col['map'])
        elif col['format'] == 'integers':
            span = col['max'] - col['min']
            cap, col['dtype'] = next((m, d) for m, d in lit._DT_MAX if span <= m)
            col['offset'] = bool(col['min'] < 0 or col['max'] > cap)
        elif col['format'] == 'strings':                    # E1 in place of uq.py:672-673
            if longest[i] > STRING_MAX:
                raise UQError('ERROR: QNAME column %d holds a token of %d bytes; a string column holds at most %d'
                              % (i + 1, longest[i], STRING_MAX))
            col['longest'] = longest[i]
            col['dtype'] = '|S%d' % max(longest[i], 1)
    return columns


def pass4(lines, total, prefix, suffix, separators, columns):
    """uq_literal.pass4 (uq.py:717-735) plus the token bytes of string columns"""
    out = [numpy.zeros(total, dtype=c['dtype']) for c in columns]
    for r, toks in enumerate(lit.qname_tokens(lines, total, prefix, suffix, separators)):
        for i, tok in enumerate(toks):
            c = columns[i]
            if c['format'] == 'mapping':
                out[i][r] = bisect.bisect_left(c['map'], tok)          # uq.py:724
            elif c['format'] == 'strings':
                out[i][r] = tok.encode('latin-1')                       # E1: zero padded by numpy
            elif c['offset']:
                out[i][r] = int(tok) - c['min']                         # uq.py:725
            else:
                out[i][r] = int(tok)                                    # uq.py:726
    return out


def _mix_qname_strings(out, cols, columns, order, raw):
    n = len(cols[0])
    perm = numpy.lexsort(cols[::-1]) if n else numpy.zeros(0, dtype=numpy.int64)     # stable argsort of the rows
    if raw:
        if order is False:
            order = perm                                                # uq.py:816 + S10
        for c, meta in zip(cols, columns):
            out[meta['name'] + '.raw'] = c[order] if isinstance(order, numpy.ndarray) else c
        return order if isinstance(order, numpy.ndarray) else None
    new = numpy.zeros(n, dtype=bool)                                    # first row of every group of equal rows
    if n:
        new[0] = True
        for c in cols:
            s = c[perm]
            new[1:] |= s[1:] != s[:-1]
    key = numpy.empty(n, dtype=numpy.int64)
    key[perm] = numpy.cumsum(new) - 1                                   # numpy.unique(return_inverse), uq.py:830
    key = key.astype(numpy.min_scalar_type(int(key.max()) if n else 0))   # uq.py:832
    if order is False:
        order = numpy.argsort(key, kind='stable')                       # uq.py:833 + S10
    out['QNAME.key'] = key[order] if isinstance(order, numpy.ndarray) else key
    first = perm[new]
    for c, meta in zip(cols, columns):
        out[meta['name']] = c[first].astype(meta['dtype'])              # uq.py:846-847
    return order if isinstance(order, numpy.ndarray) else None


def mix_qname(out, cols, columns, order, raw):
    """encode_qname (uq.py:808-851); with string columns the rows are ordered by numpy.lexsort"""
    if any(c['format'] == 'strings' for c in columns):
        return _mix_qname_strings(out, cols, columns, order, raw)
    return lit.mix_qname(out, cols, columns, order, raw)


def run_mix(dna, qual, cols, columns, sorted_on, raw_tables, pattern):
    """uq_literal.run_mix (uq.py:739-753) with this module's mix_qname"""
    out = {}
    pd, pq = pattern
    if sorted_on in ('DNA', 'QUAL'):
        first = (dna, 'DNA', pd) if sorted_on == 'DNA' else (qual, 'QUAL', pq)
        second = (qual, 'QUAL', pq) if sorted_on == 'DNA' else (dna, 'DNA', pd)
        order = lit.mix_dna_qual(out, first[0], first[1], False, first[1] in raw_tables, first[2])
        lit.mix_dna_qual(out, second[0], second[1], order, second[1] in raw_tables, second[2])
        mix_qname(out, cols, columns, order, 'QNAME' in raw_tables)
    elif sorted_on == 'QNAME':
        order = mix_qname(out, cols, columns, False, 'QNAME' in raw_tables)
        lit.mix_dna_qual(out, dna, 'DNA', order, 'DNA' in raw_tables, pd)
        lit.mix_dna_qual(out, qual, 'QUAL', order, 'QUAL' in raw_tables, pq)
    else:
        mix_qname(out, cols, columns, None, 'QNAME' in raw_tables)
        lit.mix_dna_qual(out, dna, 'DNA', None, 'DNA' in raw_tables, pd)
        lit.mix_dna_qual(out, qual, 'QUAL', None, 'QUAL' in raw_tables, pq)
    return out


def encode(fastq, sort=None, raw=None, pattern=None, pad=False, notricks=False):
    """uq_literal.encode with E1: FASTQ bytes -> (members, config)"""
    sort, raw, pattern = lit.normalise_options(sort, raw, pattern)
    lines, total = lit.split_lines(fastq)
    p1 = lit.pass1(lines, total)
    dec = lit.decide(p1, notricks=notricks, pad=pad)
    columns = pass2(lines, total, p1['prefix'], p1['suffix'], dec['separators'])
    dna, qual = lit.pass3(lines, total, dec)
    cols = pass4(lines, total, p1['prefix'], p1['suffix'], dec['separators'], columns)
    members = run_mix(dna, qual, cols, columns, sort, raw, pattern)
    config = {                                                            # uq.py:681-696, 898-900
        'base_distribution': dec['base_distribution'], 'qual_distribution': dec['qual_distribution'],
        'reads': total, 'bases': dec['bases'], 'qualities': dec['qualities'],
        'variable_read_lengths': dec['variable_read_lengths'], 'bits_per_base': dec['bits_per_base'],
        'bits_per_quality': dec['bits_per_quality'], 'N_qual': dec['N_qual'], 'dna_max': dec['dna_max'],
        'QNAME_prefix': p1['prefix'], 'QNAME_suffix': p1['suffix'], 'QNAME_separators': dec['separators'],
        'QNAME_columns': columns, 'sort': sort, 'raw': list(raw), 'pattern': pattern,
    }
    return members, config


def decode(members, config):
    """uq_literal.decode (uq.py:926-1060) with E1: members/config as read_container returns them -> FASTQ bytes"""
    pat = config['pattern']

    def table(name, p):
        if name + '.raw' in members:
            return lit.undo_pattern(members[name + '.raw'], p)
        if name in members and name + '.key' in members:
            return lit.undo_pattern(members[name], p)[members[name + '.key']]     # uq.py:953, 957
        raise UQError('ERROR: No %s data was found in this uQ file?!' % name)
    dna_t, qual_t = table('DNA', pat[0]), table('QUAL', pat[1])
    ncol = len(config['QNAME_columns'])
    if 'QNAME.key' in members:                                              # uq.py:962-973 (+S11), column by column
        qcols = [members['QNAME_%d' % (i + 1)][members['QNAME.key']] for i in range(ncol)]
    else:
        qcols = [members['QNAME_%d.raw' % (i + 1)] for i in range(ncol)]

    bases, quals = config['bases'], config['qualities']
    back = dict((v, k) for k, v in config['N_qual'].items())                # uq.py:999
    var = config['variable_read_lengths']
    nsym = var + config['dna_max']
    bb, bq = config['bits_per_base'], config['bits_per_quality']
    seps, cols = config['QNAME_separators'], config['QNAME_columns']
    out = []
    for r, (d_row, q_row) in enumerate(zip(dna_t, qual_t)):
        ds = lit._symbols(d_row, nsym * bb, bb)
        qs = lit._symbols(q_row, nsym * bq, bq)
        dna, qual = [], []
        for d, q in zip(ds, qs):                                            # uq.py:1034-1037
            qual.append(quals[q])
            dna.append(back[q] if q in back else bases[d])
        if var:                                                             # uq.py:1039-1041
            dna = dna[1 + dna.index(bases[1]):]
            qual = qual[1 + qual.index(quals[1]):]
        name = config['QNAME_prefix']                                       # uq.py:1010-1024
        for i, c in enumerate(cols):
            v = qcols[i][r]
            if c['format'] == 'mapping':
                name += c['map'][int(v)]
            elif c['format'] == 'strings':
                name += bytes(v).decode('latin-1')                         # numpy drops the zero padding
            elif c['offset']:
                name += str(int(v) + c['min'])
            else:
                name += str(int(v))
            if i < len(seps):
                name += seps[i]
        name += config['QNAME_suffix']
        out.append(name + '\n' + ''.join(dna) + '\n+\n' + ''.join(qual) + '\n')   # uq.py:1042-1045
    return ''.join(out).encode('latin-1')
