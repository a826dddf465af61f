#!/usr/bin/env python3
"""Diagnostics: grouping the rows of a packed table by destination rank (multi-GPU sample sort) on one device,
partition_positions + scatter_rows_segmented, per kernel, for 2 and 8 destinations."""
import json, os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from uq_b200 import host, multigpu
from uq_b200.device import Context

n = int(sys.argv[1]) if len(sys.argv) > 1 else 100_000_000
ctx = Context(0)
dev = ctx.synth("genome", n, 150, 1002, genome=10_000_000, pool=max(1, n // 5))
fq = ctx.adopt_fastq(dev)
p = host.prepare(ctx, fq)
out = {}
for name in ("dna", "qual"):
    t = p[name]
    for world in (2, 8):
        samples = multigpu._sample_rows(ctx, t, 1024)
        keys = np.sort(multigpu.row_key64(multigpu.pick_splitters(samples, world)))
        for it in range(2):
            ctx.sync(); ctx.timing(True); ctx.timing_reset()
            pos, counts = ctx.partition_positions(t, keys)
            buf, offs = ctx.scatter_rows_segmented(t, pos, counts, 128)
            pos.free()
            ctx.sync()
            rep = ctx.timing_report()
            buf.free()
        out["%s W=%d" % (name, world)] = {"ms": round(sum(v[1] for v in rep.values()), 3),
                                          "kernels": {k: round(v[1], 3) for k, v in rep.items() if v[1] > 0.05}}
print(json.dumps(out, indent=1))
