"""Cost of 'strings' QNAME columns (E1): 100 M x 150 bp reads of synth kind 4 (umi: the illumina header + '_<UMI>', one
string column of 6-12 bytes) against kind 0 (illumina: integer columns only), same seed, in one process, alternated.

For each input and each run (--sort DNA keyed, as bench.py; --sort QNAME keyed) it records the encode step time
(CUDA events on the context's stream, the FASTQ resident in HBM), the decode time of the container that step made,
and the uqb_ctx_timing_report rows of the string-column writer and the columns <-> rows kernels (from a separate
timed pass: per-kernel timing adds events around every launch).  The GPU name and power limit are read in the same run.

    python tools/bench_qname_strings.py [--reads 100000000] [--reps 3] [--out profiles/r04_qname_strings_100m.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# report rows kept: the string-column writer, the integer / rank column writers and tokeniser next to it, and every
# columns <-> rows kernel (the staged *_mixed pair runs when a string column is present)
KERNELS = ("k_encode_str", "k_encode_int", "k_encode_rank", "k_qname_tokens", "k_cols_to_rows", "k_rows_to_cols")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True)
    name, power, clock = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=100_000_000)
    ap.add_argument("--length", type=int, default=150)
    ap.add_argument("--seed", type=int, default=20260)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_qname_strings_100m.json"))
    a = ap.parse_args()
    from uq_b200 import host
    from uq_b200.device import Context
    ctx = Context(0)
    kinds = ("umi", "illumina")
    src = {k: ctx.synth(k, a.reads, a.length, a.seed) for k in kinds}
    fqs = {k: ctx.adopt_fastq(src[k]) for k in kinds}
    runs = (("DNA", "sort DNA keyed"), ("QNAME", "sort QNAME keyed"))

    def step(kind, sort):
        ctx.sync()
        ctx.span_begin()
        dm, cfg = host.encode_device(ctx, fqs[kind], sort=sort)
        enc = ctx.span_end()
        ctx.span_begin()
        text = host.decode_members_device(ctx, dm, cfg)
        dec = ctx.span_end()
        nbytes = text.nbytes
        text.free(); dm.free()
        return enc, dec, nbytes, cfg

    out = dict(gpu=gpu_info(), reads=a.reads, length=a.length, seed=a.seed, reps=a.reps, runs={})
    for kind in kinds:                          # warm-up of every shape
        for sort, _ in runs:
            step(kind, sort)
    for rep in range(a.reps):                   # alternated: umi, illumina, umi, ...
        for sort, label in runs:
            for kind in kinds:
                enc, dec, nbytes, cfg = step(kind, sort)
                r = out["runs"].setdefault("%s %s" % (kind, label), dict(step_ms=[], decode_ms=[]))
                r["step_ms"].append(round(enc, 3))
                r["decode_ms"].append(round(dec, 3))
                r["fastq_bytes"] = nbytes
                r["qname_columns"] = [dict((k, c[k]) for k in ("format", "dtype")) for c in cfg["QNAME_columns"]]
    ctx.timing(True)
    for sort, label in runs:
        for kind in kinds:
            ctx.timing_reset()
            step(kind, sort)
            rep = ctx.timing_report()
            rows = {k: dict(launches=v[0], ms=round(v[1], 3), algorithmic_bytes=v[2]) for k, v in rep.items()
                    if any(s in k for s in KERNELS)}
            out["runs"]["%s %s" % (kind, label)]["kernels"] = rows
    ctx.timing(False)
    for r in out["runs"].values():
        r["step_ms_median"] = sorted(r["step_ms"])[len(r["step_ms"]) // 2]
        r["decode_ms_median"] = sorted(r["decode_ms"])[len(r["decode_ms"]) // 2]
    for k in kinds:
        fqs[k].free(); src[k].free()
    ctx.close()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print(json.dumps({k: (v["step_ms_median"], v["decode_ms_median"]) for k, v in out["runs"].items()}))


if __name__ == "__main__":
    main()
