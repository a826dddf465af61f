"""Cost of one-column QNAMEs (E2): 100 M x 150 bp reads of synth kind 5 (renamed: @SRR0000001.<n>, --sort QNAME keyed)
and kind 6 (mixed CASAVA / pre-1.8 headers, everything raw), next to kind 0 (illumina, --sort DNA keyed as bench.py),
same seed, in one process.

For each input it records
  - the encode step and the decode of the container it made (CUDA events on the context's stream, FASTQ resident in HBM,
    every run warmed up once, then `--reps` runs alternated over the inputs);
  - per stage of prepare / run_mix, from a separate pass with per-kernel timing on: the CUDA-event time of every kernel
    launched in that stage ('qname_remainder' is the extra tokeniser pass that measures the shortest remainder, which
    only E2 files run; 'qname_scan' counts every tokeniser pass with its column statistics).
The GPU name and power limit are read in the same run.

    python tools/profile_qname_fallback.py [--reads 100000000] [--reps 3] [--out profiles/r05_qname_fallback_100m.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

RUNS = (("renamed", dict(sort="QNAME"), "renamed sort QNAME keyed"),
        ("mixed", dict(sort="None", raw=["DNA", "QUAL", "QNAME"]), "mixed raw"),
        ("illumina", dict(sort="DNA"), "illumina sort DNA keyed"))


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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_qname_fallback_100m.json"))
    a = ap.parse_args()
    from uq_b200 import host
    from uq_b200.device import Context
    ctx = Context(0)
    out = dict(gpu=gpu_info(), reads=a.reads, length=a.length, seed=a.seed, reps=a.reps, runs={})

    def step(fq, kw):
        ctx.sync()
        ctx.span_begin()
        dm, cfg = host.encode_device(ctx, fq, **kw)
        enc = ctx.span_end()
        ctx.span_begin()
        text = host.decode_members_device(ctx, dm, cfg)
        dec = ctx.span_end()
        nbytes = text.nbytes
        text.free(); dm.free()
        return enc, dec, nbytes, cfg

    for kind, kw, label in RUNS:
        # one input at a time in HBM: the three FASTQs and their encodes together would not leave room to spare
        src = ctx.synth(kind, a.reads, a.length, a.seed)
        fq = ctx.adopt_fastq(src)
        step(fq, kw)                                    # warm-up of every shape
        r = out["runs"][label] = dict(step_ms=[], decode_ms=[])
        for _ in range(a.reps):
            enc, dec, nbytes, cfg = step(fq, kw)
            r["step_ms"].append(round(enc, 3))
            r["decode_ms"].append(round(dec, 3))
        r["fastq_bytes"] = nbytes
        r["qname_layout"] = dict(prefix=cfg["QNAME_prefix"], suffix=cfg["QNAME_suffix"],
                                 separators=cfg["QNAME_separators"],
                                 columns=[dict((k, c[k]) for k in ("format", "dtype")) for c in cfg["QNAME_columns"]])
        r["step_ms_median"] = sorted(r["step_ms"])[len(r["step_ms"]) // 2]
        r["decode_ms_median"] = sorted(r["decode_ms"])[len(r["decode_ms"]) // 2]
        ctx.timing(True)
        ctx.timing_reset()
        host.PHASE_LOG, host.PHASE_KERNELS = {}, {}
        step(fq, kw)
        r["stages"] = {ph: dict(kernel_ms=round(sum(v[1] for v in ks.values()), 3),
                                kernels={k: dict(launches=v[0], ms=round(v[1], 3)) for k, v in sorted(ks.items())})
                       for ph, ks in host.PHASE_KERNELS.items()}
        host.PHASE_LOG = host.PHASE_KERNELS = None
        ctx.timing(False)
        fq.free(); src.free()
    ctx.close()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print(json.dumps({k: (v["step_ms_median"], v["decode_ms_median"],
                          {ph: s["kernel_ms"] for ph, s in v["stages"].items() if ph.startswith("qname")})
                      for k, v in out["runs"].items()}))


if __name__ == "__main__":
    main()
