"""Cost of --verify (host.verify_device) next to the encode it checks, in one process:
  - configs[1]: 100 M x 150 bp, --sort DNA keyed (the bench's encode), and the same reads raw and unsorted;
  - configs[4]: 1 M reads of 1-20 kb, --sort QUAL.

For each input it records
  - the encode step and the verify of its members (CUDA events on the context's stream, FASTQ resident in HBM, warmed
    up once, then `--reps` runs), with the default batch of 2^24 rows (or fewer when memory says so);
  - from a separate pass with per-kernel timing on: the CUDA-event time of every kernel per verify phase (verify_perm:
    permutation check; verify_rows: keys widened and rows gathered for a batch; verify_decode; verify_split: line offsets
    of the decoded text; verify_compare: k_verify_records), summed over the batches and per batch;
  - the compare kernel's algorithmic bytes (both texts, the line offsets, the order) over its time, against the HBM
    roofline of DESIGN section 3 (6544.7 GB/s measured) and the data-sheet 7.7 TB/s.
The GPU name and power limit are read in the same run.

    python tools/profile_verify.py [--reps 3] [--out profiles/r06_verify_100m.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_MEASURED_GBS = 6544.7
HBM_DATASHEET_GBS = 7700.0


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True)
    name, power, clock = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=100_000_000)
    ap.add_argument("--ont-reads", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_verify_100m.json"))
    a = ap.parse_args()
    from oracle import synth
    from uq_b200 import host
    from uq_b200.device import Context
    ctx = Context(0)
    out = dict(gpu=gpu_info(), reps=a.reps, hbm_roofline_gbs=HBM_MEASURED_GBS, runs={})

    def make_illumina():
        return ctx.synth("genome", a.reads, 150, 1002, genome=10_000_000, pool=a.reads // 5)

    def make_ont():
        return ctx.synth("ont", a.ont_reads, (1000, 20000), 1005, len_table=synth.ont_length_table(1000, 20000))
    inputs = (("configs[1] sort DNA keyed", make_illumina, [("configs[1] sort DNA keyed", dict(sort="DNA")),
                                                            ("configs[1] raw unsorted", dict(sort="None", raw=["DNA", "QUAL", "QNAME"]))]),
              ("configs[4]", make_ont, [("configs[4] 1-20 kb sort QUAL", dict(sort="QUAL"))]))

    def step(fq, kw):
        ctx.sync()
        ctx.span_begin()
        dm, cfg = host.encode_device(ctx, fq, **kw)
        enc = ctx.span_end()
        batch = host.verify_batch_rows(ctx, fq, dm, cfg)
        ctx.span_begin()
        rep = host.verify_device(ctx, fq, dm, cfg, batch_rows=batch)
        ver = ctx.span_end()
        assert host.verify_clean(rep) and rep["records"] == cfg["reads"], rep
        dm.free()
        return enc, ver, batch

    for _, make, runs in inputs:
        src = make()
        fq = ctx.adopt_fastq(src)
        for label, kw in runs:
            step(fq, kw)                                        # warm-up of every shape
            r = out["runs"][label] = dict(encode_ms=[], verify_ms=[], fastq_bytes=src.nbytes, options=kw)
            for _ in range(a.reps):
                enc, ver, batch = step(fq, kw)
                r["encode_ms"].append(round(enc, 3))
                r["verify_ms"].append(round(ver, 3))
            r["batch_rows"] = batch
            r["batches"] = -(-fq.n_reads // batch)
            r["encode_ms_median"] = sorted(r["encode_ms"])[len(r["encode_ms"]) // 2]
            r["verify_ms_median"] = sorted(r["verify_ms"])[len(r["verify_ms"]) // 2]
            # per-kernel pass: phases of verify_device, kernel times summed over the batches
            dm, cfg = host.encode_device(ctx, fq, **kw)
            ctx.timing(True)
            ctx.timing_reset()
            host.PHASE_LOG, host.PHASE_KERNELS = {}, {}
            host.verify_device(ctx, fq, dm, cfg, batch_rows=batch)
            rep = ctx.timing_report()
            r["phases"] = {ph: dict(kernel_ms=round(sum(v[1] for v in ks.values()), 3),
                                    kernel_ms_per_batch=round(sum(v[1] for v in ks.values()) / r["batches"], 3),
                                    wall_ms_with_syncs=round(host.PHASE_LOG[ph], 3),
                                    kernels={k: dict(launches=v[0], ms=round(v[1], 3)) for k, v in sorted(ks.items())})
                           for ph, ks in host.PHASE_KERNELS.items()}
            host.PHASE_LOG = host.PHASE_KERNELS = None
            ctx.timing(False)
            dm.free()
            launches, ms, nbytes = rep["k_verify_records"]
            gbs = nbytes / (ms * 1e-3) / 1e9
            r["compare"] = dict(launches=launches, ms=round(ms, 3), algorithmic_bytes=nbytes, gbs=round(gbs, 1),
                                of_measured_roofline=round(gbs / HBM_MEASURED_GBS, 3),
                                of_datasheet=round(gbs / HBM_DATASHEET_GBS, 3))
            if "k_perm_mark" in rep:
                r["permutation_check_ms"] = round(rep["k_perm_mark"][1] + rep["k_perm_missing"][1], 3)
        fq.free(); src.free()
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print(json.dumps({"gpu": out["gpu"], "runs": {k: dict(encode=v["encode_ms_median"], verify=v["verify_ms_median"], batches=v["batches"],
                                                          compare=v["compare"],
                                                          phases={p: s["kernel_ms"] for p, s in v["phases"].items()})
                                                  for k, v in out["runs"].items()}}, indent=1))


if __name__ == "__main__":
    main()
