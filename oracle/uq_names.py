"""Declared extension E2 (DESIGN section 4) on top of the literal oracle: QNAMEs stored as one column.

TEST INFRASTRUCTURE.  The reference cannot cut every file's QNAMEs into columns: with no separator (Q6), separators in
a different order ("so unusual/improbable"), a name shorter than the running common prefix or suffix (Q8, IndexError)
or a separator class that breaks its unescaped regex (Q11) it stops.  The B200 path also stops the reference's layout
where a record does not hold the separators in their order.  On exactly those files E2 stores

  layout      prefix = the longest common prefix of all names, suffix = the longest common suffix of the remainders
              name[len(prefix):], separators = '', one column QNAME_1 = the rest of every name
  typing      uq.py:586-676 on that one column, except that it is 'integers' only when every token is the canonical
              text of an int64 (str(int(t)) == t); a demoted column that is not is 'strings' (E1)
  Pass 4      integers (minus min with offset), mapping ranks, or the token bytes
  mixes       uq_strings.run_mix (lexsort order for a string column, the reference's own otherwise)
  decode      uq_strings.decode: prefix + token + suffix

Every record is walked in plain Python; nothing here is taken from uq_b200.  Every other file is encoded by
uq_strings.encode, which on files without string columns is uq_literal.encode.
"""
import bisect
import collections
import re

import numpy

from . import uq_literal as lit
from . import uq_strings
from .uq_literal import UQError

INT64 = (-2 ** 63, 2 ** 63 - 1)


def names_of(lines, total):
    return [lines[4 * r] for r in range(total)]


def reference_layout(lines, total):
    """(prefix, suffix, separators) when the file's QNAMEs split into the reference's columns, None when E2 applies.
    The separators can be '' (no surviving separator occurs in the first and the last name): such a file is stored as
    one column under the reference's own layout and typing, and is not E2's."""
    try:
        p1 = lit.pass1(lines, total)
        dec = lit.decide(p1)
    except (UQError, IndexError, re.error):                    # Q6, order, Q8, Q11 (a class that does not compile)
        return None
    prefix, suffix, seps = p1['prefix'], p1['suffix'], dec['separators']
    if any(ch in '-^]\\' for ch in p1['sep_count']):           # Q11: the unescaped class means something else
        meant = ''.join(re.escape(ch) for ch in p1['sep_count'])
        for name in (p1['last_name'], p1['first_name']):
            if ''.join(re.findall('([' + meant + ']+)', name[len(prefix):-1 - len(suffix)])) != seps:
                return None
    sepset = set(seps)
    for name in names_of(lines, total):                        # every record holds the separators in their order
        mid = name[len(prefix):len(name) - len(suffix)] if len(name) - len(suffix) > len(prefix) else ''
        if ''.join(ch for ch in mid if ch in sepset) != seps:
            return None
    return prefix, suffix, seps


def layout(lines, total):
    """E2: (prefix, suffix) from every name"""
    names = names_of(lines, total)
    prefix = names[0]
    for name in names[1:]:
        k = 0
        while k < min(len(prefix), len(name)) and prefix[k] == name[k]:
            k += 1
        prefix = prefix[:k]
    rest = [name[len(prefix):] for name in names]
    suffix = rest[0]
    for r in rest[1:]:
        k = 0
        while k < min(len(suffix), len(r)) and suffix[len(suffix) - 1 - k] == r[len(r) - 1 - k]:
            k += 1
        suffix = suffix[len(suffix) - k:]
    return prefix, suffix


def tokens(lines, total, prefix, suffix):
    return [name[len(prefix):len(name) - len(suffix)] for name in names_of(lines, total)]


def canonical_int(tok):
    try:
        v = int(tok)
    except ValueError:
        return None
    return v if str(v) == tok and INT64[0] <= v <= INT64[1] else None


def pass2(toks):
    """uq.py:604-676 on the single column, with E2's integer rule"""
    col = {'name': 'QNAME_1', 'format': 'mapping', 'map': set()}
    target = 10000
    last = -1
    for last, tok in enumerate(toks):                          # uq.py:614-636
        if col['format'] == 'mapping':
            col['map'].add(tok)
        if last == target:
            if col['format'] == 'mapping' and len(col['map']) > last // 10:
                col['format'] = 'demoted'
                del col['map']
            target *= 2
    if col['format'] == 'mapping' and len(col['map']) > last // 10:      # uq.py:638
        col['format'] = 'demoted'
        del col['map']
    vals = [canonical_int(t) for t in toks]
    exact = all(v is not None for v in vals)
    if col['format'] == 'demoted':
        if exact:
            col['format'] = 'integers'
            col['min'], col['max'] = min(vals), max(vals)
            cap, col['dtype'] = next((m, d) for m, d in lit._DT_MAX if col['max'] - col['min'] <= m)
            col['offset'] = bool(col['min'] < 0 or col['max'] > cap)
        else:
            longest = max(len(t) for t in toks)
            if longest > uq_strings.STRING_MAX:
                raise UQError('ERROR: QNAME column 1 holds a token of %d bytes; a string column holds at most %d'
                              % (longest, uq_strings.STRING_MAX))
            col['format'] = 'strings'
            col['longest'] = longest
            col['dtype'] = '|S%d' % max(longest, 1)
    else:                                                      # uq.py:643-661
        cap, col['dtype'] = next((m, d) for m, d in lit._DT_MAX if len(col['map']) <= m)
        if exact and max(vals) - min(vals) <= cap:
            col['format'] = 'integers'
            col['max'], col['min'] = max(vals), min(vals)
            col['offset'] = bool(col['min'] < 0 or col['max'] > cap)
            del col['map']
        else:
            col['map'] = sorted(col['map'])
    return [col]


def pass4(toks, columns):
    c = columns[0]
    out = numpy.zeros(len(toks), dtype=c['dtype'])
    for r, tok in enumerate(toks):
        if c['format'] == 'mapping':
            out[r] = bisect.bisect_left(c['map'], tok)                 # uq.py:724
        elif c['format'] == 'strings':
            out[r] = tok.encode('latin-1')
        else:
            out[r] = int(tok) - (c['min'] if c['offset'] else 0)       # uq.py:725-726
    return [out]


def alphabets(lines, total, notricks=False, pad=False):
    """uq.py:338-545 without the QNAME part: the reference's own decide() run on the sequence statistics alone (its
    separator step, handed an empty name pair and a separator that occurs nowhere, yields '')"""
    joint = {}
    lo = hi = len(lines[1])
    for r in range(total):
        seq, plus, qual = lines[4 * r + 1], lines[4 * r + 2], lines[4 * r + 3]
        if plus[:1] != '+':
            raise UQError('ERROR: For entry %d the third line does not start with +' % r)
        if len(seq) != len(qual):
            raise UQError('ERROR: Length of DNA does not match the length of the quality scores for entry %d' % (r + 1))
        lo, hi = min(lo, len(seq)), max(hi, len(seq))
        for b, q in zip(seq, qual):
            joint.setdefault(b, collections.defaultdict(int))[q] += 1
    p1 = dict(prefix='', suffix='', sep_count={'\n': 1}, first_name='', last_name='', dna_min=lo, dna_max=hi, joint=joint)
    dec = lit.decide(p1, notricks=notricks, pad=pad)
    assert dec['separators'] == ''
    return dec


def encode(fastq, sort=None, raw=None, pattern=None, pad=False, notricks=False, stages=None):
    """FASTQ bytes -> (members, config): uq_strings.encode where the reference's layout holds, E2 everywhere else"""
    lines, total = lit.split_lines(fastq)
    if total and not lines[0].startswith('@'):
        raise UQError('ERROR: This does not look like a FASTA/FASTQ file! (first line does not start with @)')
    if reference_layout(lines, total) is not None:
        return uq_strings.encode(fastq, sort=sort, raw=raw, pattern=pattern, pad=pad, notricks=notricks)
    sort, raw, pattern = lit.normalise_options(sort, raw, pattern)
    dec = alphabets(lines, total, notricks=notricks, pad=pad)
    prefix, suffix = layout(lines, total)
    toks = tokens(lines, total, prefix, suffix)
    columns = pass2(toks)
    dna, qual = lit.pass3(lines, total, dec)
    cols = pass4(toks, columns)
    if stages is not None:
        stages.update(prefix=prefix, suffix=suffix, columns=columns, tokens=toks)
    members = uq_strings.run_mix(dna, qual, cols, columns, sort, raw, pattern)
    config = {
        'base_distribution': dec['base_distribution'], 'qual_distribution': dec['qual_distribution'],
        'reads': total, 'bases': dec['bases'], 'qualities': dec['qualities'],
        'variable_read_lengths': dec['variable_read_lengths'], 'bits_per_base': dec['bits_per_base'],
        'bits_per_quality': dec['bits_per_quality'], 'N_qual': dec['N_qual'], 'dna_max': dec['dna_max'],
        'QNAME_prefix': prefix, 'QNAME_suffix': suffix, 'QNAME_separators': '',
        'QNAME_columns': columns, 'sort': sort, 'raw': list(raw), 'pattern': pattern,
    }
    return members, config


decode = uq_strings.decode
