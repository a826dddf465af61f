#!/usr/bin/env python3
"""uq.py on a B200: the reference's command line (uq.py:21-34), option checks (uq.py:52-71) and container
format, with the FASTQ -> uQ encode and uQ -> FASTQ decode hot path running on the GPU through
libuqb200.so.  Host logic only; there is no CPU implementation of the path in this package.

    python -m uq_b200.uq -i reads.fastq [--sort DNA|QUAL|QNAME|None] [--raw DNA QUAL QNAME] \\
                         [--pattern 0.1 0.1] [--pad] [--notricks] [--peek] [--test] [--compressor CMD] [--verify]
    python -m uq_b200.uq -i reads.fastq.uQ --decode > reads.fastq
"""
import argparse
import io
import json
import os
import subprocess
import sys
import time

import numpy

from . import container, host
from .device import Context

ALL_RAW = [('DNA', 'QUAL', 'QNAME'), ('DNA', 'QUAL'), ('QUAL', 'QNAME'), ('DNA', 'QNAME'), ('DNA',), ('QUAL',), ('QNAME',), (None,)]


def build_parser():
    p = argparse.ArgumentParser(description="This tool converys FASTQ files to microq (uQ) files and back (B200 device path).")
    p.add_argument("-i", "--input", required=True, help='Required. Input FASTQ/uQ file path.')
    p.add_argument("-o", "--output", help='Optional. FASTQ->uQ only. Default is to append .uQ to input filename.')
    p.add_argument("--compressor", action='store', help='Optional. Path to compression program that accepts data on stdin and prints to stdout/pipe)')
    p.add_argument("--sort", action='store', help='Optional. [DNA/QUAL/QNAME/None] Resort FASTQ. See output of --test for optimium method.')
    p.add_argument("--raw", nargs='+', metavar='file name', help='Optional. [DNA/QUAL/QNAME/None] Store tables raw rather than unique & sorted + key.')
    p.add_argument("--pattern", nargs='+', metavar='pattern', help='Optional. [0.1/0.2/1.1/1.2/2.1/2.2/3.1/3.2] x2 (DNA|QUAL)')
    p.add_argument("--temp", help='Optional. Kept for compatibility; this implementation needs no temporary files.')
    p.add_argument("--test", action='store_true', default=False, help='Optional. Try all sort/raw/pattern combinations (search loop stays on the CPU).')
    p.add_argument("--notricks", action='store_true', default=False, help='Optional. Prevents conversion of N to the most popular base.')
    p.add_argument("--pad", action='store_true', default=False, help='Optional. Pads DNA/QUAL to the nearest 2/4/8 bits.')
    p.add_argument("--peek", action='store_true', default=False, help='Optional. No output files are created, the input is just scanned and report printed to terminal.')
    p.add_argument("--decode", action='store_true', default=False, help='Requred if you want to convert a .uQ back to .fastq')
    p.add_argument("--device", type=int, default=0, help='CUDA device ordinal (this implementation only).')
    p.add_argument("--verify", action='store_true', default=False,
                   help='Optional. FASTQ->uQ only. Decode the container on the GPU and compare every record with its input '
                        'record before writing it; on any difference nothing is written and the exit status is 1.')
    return p


def check_options(args):
    if args.verify and (args.decode or args.peek):
        raise host.UQError('ERROR: --verify checks a FASTQ -> uQ encode; it cannot be combined with --%s'
                           % ('decode' if args.decode else 'peek'))


HINTS = {0: 'integer QNAME columns lose leading zeros and "+" signs in the reference format (Q9)',
         2: 'the reference format keeps no text after the "+" of the third line (Q13)'}


def verify_failure(report):
    """the report of a verify that found differences -> the lines to print"""
    out = ['ERROR: --verify: the container does not reproduce the input; nothing was written.']
    for f, field in enumerate(host.FIELDS):
        if not report['differ'][f]:
            continue
        out.append('  %s: %d records differ; first at container row %d, input record %d' % (
            field, report['differ'][f], report['first_row'][f], report['first_src'][f]))
        want, got = report['lines'].get(f, (None, None))
        if want is not None:
            out.append('    input:   %r' % want)
        if got is not None:
            out.append('    decoded: %r' % got)
        if f in HINTS:
            out.append('    hint: ' + HINTS[f])
    if report['missing'] >= 0:
        out.append('  order: input record %d is missing from the container' % report['missing'])
    return out


def compressed_size(arr, compressor):
    """uq.py:277-285: size of the NPY stream after the external compressor (CPU, excluded from timing)."""
    if not compressor:
        return arr.nbytes
    r = subprocess.run(compressor + ' | wc -c', shell=True, input=container.npy_bytes(arr), stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
    return int(r.stdout.split()[0])


def run_test_search(ctx, fq_bytes, args):
    """The --test loop (uq.py:855-889).  The FASTQ is loaded and Pass 1-4 run ONCE; host.MixFeed keeps the packed tables
    and at most one sort per table in HBM and serves every candidate member as a gather / layout of those (SURVEY
    section 8 f1).  The compressor and the argmin stay on the CPU exactly as in the reference."""
    fq = ctx.load_fastq(fq_bytes)
    feed = host.MixFeed(ctx, fq, pad=args.pad, notricks=args.notricks)
    results = []
    patterns = [args.pattern[0]] if args.pattern else (host.PATTERNS if args.compressor else ['0.1'])
    raws = ALL_RAW if args.raw is None else [tuple(args.raw)]
    sorts = (['DNA', 'QUAL', 'QNAME', None] if args.compressor else [None]) if args.sort is None else [args.sort]
    sizes = {}                                       # id of the cached host array -> compressed size (members repeat between mixes)
    for raw_tables in raws:
        for to_sort in sorts:
            best = {}
            for pat in patterns:
                members = feed.members(sort=to_sort if to_sort else 'None', raw=[r if r else 'none' for r in raw_tables],
                                       pattern=[pat, pat] if not args.pattern else args.pattern)
                for name, arr in members.items():
                    key = (name, to_sort if not name.endswith(('DNA', 'QUAL')) else None, pat if name.startswith(('DNA', 'QUAL')) and not name.endswith('.key') else None)
                    if key not in sizes:
                        sizes[key] = compressed_size(arr, args.compressor)
                    size = sizes[key]
                    if name.startswith(('DNA', 'QUAL')) and not name.endswith('.key'):
                        if name not in best or size < best[name][0]:
                            best[name] = (size, pat)
                    else:
                        best[name] = (size, None)
            total = sum(v[0] for v in best.values())
            results.append(dict(total_size=total, sorted_on=to_sort, raw_tables=raw_tables, detail=best))
            print(str(total).rjust(17), str(to_sort).ljust(8), str(tuple(raw_tables)).ljust(27))
    feed.free()
    fq.free()
    win = sorted(results, key=lambda k: k['total_size'])[0]
    d = win['detail']
    pat_d = next((v[1] for k, v in d.items() if k in ('DNA', 'DNA.raw')), '0.1') or '0.1'
    pat_q = next((v[1] for k, v in d.items() if k in ('QUAL', 'QUAL.raw')), '0.1') or '0.1'
    return win['sorted_on'], win['raw_tables'], [pat_d, pat_q]


def main(argv=None):
    args = build_parser().parse_args(argv)
    if not os.path.isfile(args.input):                                                  # uq.py:71
        print('ERROR: Sorry, the input path you have specified is not a file!')
        return 0
    try:
        check_options(args)
        ctx = Context(args.device)
        if args.decode:
            members, config = container.read_container(args.input)
            out = host.decode(members, config, ctx=ctx)
            sys.stdout.buffer.write(out.tobytes())                                      # uq.py:1042-1045 (stdout, Q14)
            return 0
        if args.output is None:
            args.output = args.input + '.uQ'                                            # uq.py:75
        t0 = time.time()
        size = os.path.getsize(args.input)
        pin_in = ctx.pinned_empty(size)                                                 # the file goes straight into pinned memory
        with open(args.input, 'rb') as f:
            got = 0
            view = memoryview(pin_in.array)
            while got < size:
                k = f.readinto(view[got:])
                if not k:
                    break
                got += k
        data = pin_in.array[:got]
        sort, raw, pattern = args.sort, args.raw, args.pattern
        host.normalise_options(sort, raw, pattern)                                      # validates like uq.py:52-69
        if args.peek:                                                                   # uq.py:698-702
            fq = ctx.load_fastq(data)
            stages = {}
            members, config = host.encode_device(ctx, fq, sort='None', raw=['DNA', 'QUAL', 'QNAME'], pad=args.pad, notricks=args.notricks, stages=stages)
            for k in ('sort', 'raw', 'pattern'):
                config.pop(k)
            print('The config.json would look like:')
            print(json.dumps(config, indent=4, sort_keys=True))
            return 0
        if args.test:
            s, r, p = run_test_search(ctx, data, args)
            sort, raw, pattern = (s if s else 'None'), [x if x else 'none' for x in r], p
            print('Parameters found to be the best for this data type:\n   --sort', sort, '--raw', ' '.join(map(str, raw)), '--pattern', ' '.join(pattern))
        # H2D in chunks overlapped with the record split and the Pass-1 statistics; every member starts its device->host
        # copy into its own pinned buffer the moment it is final; the container is written from those buffers
        pins = []

        def sink(name, nbytes):
            pins.append(ctx.pinned_empty(nbytes))
            return pins[-1].array

        fq = ctx.load_fastq_streamed(data) if got >= (1 << 20) else ctx.load_fastq(data)
        dmembers, config = host.encode_device(ctx, fq, sort=sort, raw=raw, pattern=pattern, pad=args.pad, notricks=args.notricks, sink=sink)
        if args.verify:                                                                 # while the members' D2H copies run
            tv = time.time()
            batch = host.verify_batch_rows(ctx, fq, dmembers, config)
            if batch == 0:
                raise host.UQError('ERROR: --verify: not enough free device memory to decode even 2^20 records next to the encoded members')
            report = host.verify_device(ctx, fq, dmembers, config, batch_rows=batch)
            if not host.verify_clean(report):
                dmembers.free(); fq.free()
                for p in pins:
                    p.free()
                print('\n'.join(verify_failure(report)))
                return 1
            print('Verified: all %d records decode to their input records (%.3f s)' % (report['records'], time.time() - tv))
        members = dmembers.download()
        print('\nWriting final config...')
        print('Archiving results...')
        container.write_container(args.output, members, config)
        dmembers.free(); fq.free()
        for p in pins:
            p.free()
        print('All Done! :)  (%d reads, %.2f s, %d kernel launches on cuda:%d)' % (config['reads'], time.time() - t0, ctx.launches, args.device))
    except host.UQError as e:                                                           # uq.py:48-50: print, exit status 0 (a failed --verify: 1)
        print(e)
    return 0


if __name__ == '__main__':
    sys.exit(main())
