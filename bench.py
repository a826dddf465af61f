#!/usr/bin/env python3
"""bench.py - FASTQ->uQ encode throughput of the B200 path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # ours
    python bench.py ... --dump-outputs DIR                          # also: outputs of the last timed step as DIR/*.npy
    python bench.py --impl reference [--steps K] [--warmup W]      # the reference algorithm on host cores

Workload (BASELINE.json configs[1]): 100 M reads x 150 bp Illumina-style synthetic FASTQ,
`--sort DNA` with keyed (unique table + index) DNA / QUAL / QNAME tables.  One "step" is one full
encode of the whole FASTQ: record split -> Pass-1 statistics -> QNAME scan -> pack -> sort/unique ->
layout, ending with every output array resident in HBM in its final layout.

  value  reads/s with the FASTQ already resident in HBM (CUDA-event time on the context's stream,
         max over ranks).
  e2e    the same encode through the public API with HOST buffers: pinned FASTQ -> H2D -> encode ->
         D2H of every output array into pinned host memory, all inside the timed region.
  roofline  the kernel with the largest share of the step: algorithmic bytes / event time vs the
         measured HBM copy bandwidth (MEASURED_PEAKS.json).
  cpu_baseline  the oracle's literal restatement of uq.py (1 core, the reference is single threaded)
         on a bounded sample of the same FASTQ.

Multi-GPU (torchrun, one process per GPU): rank r holds the contiguous read range [r n, (r+1) n) of ONE file and the
ranks produce ONE global container (merged statistics, partition-first sample sort whose rows are stored straight into
the receivers' peer-mapped windows over NVLink - NCCL all-to-all where no window is available -, global --sort order;
DESIGN.md section 6).  `--strong` divides ONE file of --reads reads over the ranks instead.  Weak scaling: n = 100 M reads per GPU.  Before the timed
loop every N>1 run encodes a small file both ways (sharded over the ranks and whole on rank 0), compares every member
and the config, decodes the container over the ranks, and reports the outcome as `parity_check`; a mismatch ends the
run with a non-zero exit code.  `--multi shards` (independent container shards, no collective) is kept as a diagnostic.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SORT, RAW, PATTERN = "DNA", None, None          # configs[1]: --sort DNA, keyed tables, default pattern
READ_LEN = 150
GENOME = 10_000_000
SEED = 1002


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        # median over samples under load (the top half of the samples)
        load = sm[len(sm) // 2:] if sm else []
        med = load[len(load) // 2] if load else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


_REAL_STDOUT = None


def quiet_stdout():
    """Everything libraries print on fd 1 (e.g. the NCCL version banner) goes to stderr; the one JSON line is written
    to the real stdout by emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


def dump_outputs(path, arrays, budget=60_000_000):
    """arrays (name -> ndarray, the members encode hands its caller) -> path/<name>.npy, so that two builds can be compared
    value for value.  Values are float32 for 1- and 2-byte integers and float64 otherwise (exact below 2**53).  An array
    larger than its equal share of `budget` bytes is replaced by the elements at a fixed, seeded set of flat (C-order)
    indices, the same for every array of that size."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    per = budget // (8 * max(len(arrays), 1))
    for name, a in sorted(arrays.items()):
        if a.size > per:
            idx = np.sort(np.random.default_rng(SEED).choice(a.size, per, replace=False))
            a = a[np.unravel_index(idx, a.shape)]
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float32 if a.dtype.itemsize <= 2 else np.float64))


def run_ours(args):
    quiet_stdout()
    from uq_b200 import shard
    rank, local_rank, world = shard.world()
    if args.dump_outputs and world > 1:
        sys.exit("--dump-outputs: single-process runs only")
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        # the row exchange of the sample sort is one large send/recv per peer: give NCCL's point-to-point path all channels
        os.environ.setdefault("NCCL_MIN_P2P_NCHANNELS", "32")
        os.environ.setdefault("NCCL_MAX_P2P_NCHANNELS", "32")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from uq_b200 import host
    from uq_b200.device import Context
    red = shard.Reducer(dist, "cuda")
    barrier, max_over_ranks, sum_over_ranks = red.barrier, red.max, red.sum

    tstream = None
    if world > 1 and args.multi == "global":
        # the context runs on a torch stream, so that the NCCL exchanges can be ordered against it on the device
        tstream = torch.cuda.Stream(device=local_rank)
        ctx = Context(local_rank, stream=tstream.cuda_stream)
    else:
        ctx = Context(local_rank)
    n = args.reads
    # weak scaling keeps the per-GPU work fixed: the genome and the quality pool grow with the total number of reads, so
    # that the duplication structure of the file (reads per genome position, reads per quality string) stays that of
    # configs[1] - with a fixed 10 Mbp genome an N-GPU file would hold N times as many copies of every read
    genome = GENOME * world
    pool = max(1, n * world // 5)
    if args.strong and world > 1:
        # strong scaling (diagnostics, profiles/): ONE configs[1] file of --reads reads in total, 1/N of it per GPU
        genome, pool = GENOME, max(1, n // 5)
        n = n // world
    first, n = shard.shard_range(rank, world, n)
    dev = ctx.synth("genome", n, READ_LEN, SEED, first=first, genome=genome, pool=pool)
    fbytes = dev.nbytes
    opts = dict(sort=SORT, raw=RAW, pattern=PATTERN)

    global_mode = world > 1 and args.multi == "global"
    if global_mode:
        from uq_b200 import multigpu
        comm = multigpu.Comm(dist, "cuda:%d" % local_rank, stream=tstream)
        if not args.no_p2p:
            # receive slots every rank can store into (symmetric memory): 3 slots, each holding the largest table a rank can
            # receive (113-byte QUAL rows, 30 % skew margin).  A table that does not fit goes through NCCL instead.
            try:
                slot = int(1.3 * n * 128)
                comm.window = multigpu.open_peer_window(dist, "cuda:%d" % local_rank, tstream, 3 * slot, slots=3)
                exchange = "peer window (symmetric memory, %d x %.1f GB per rank): rows stored into the receivers' memory by uqb_scatter_rows_to" % (3, slot / 1e9)
                # measured at N=2 (profiles/README.md): running the exchange on a side stream next to the sort of the previous
                # table gains nothing - the stores compete with the sort for the memory system (183.6 / 187.3 ms against
                # 182.3 ms serial) and the copy engines move peer data too slowly (187.8 ms) - so both stay opt-in
                side = os.environ.get("UQB_MG_SIDE", "0")
                if side == "dma":
                    comm.side = torch.cuda.Stream(device=local_rank, priority=-1)
                    comm.exchange_mode = "dma"
                    exchange = ("peer window (symmetric memory, %d x %.1f GB per rank): rows grouped by destination in local HBM "
                                "(uqb_scatter_rows_segmented), segments pushed into the receivers' memory by the copy engines on a "
                                "side stream, under the sort of the previous table" % (3, slot / 1e9))
                elif side == "stores":
                    comm.side = torch.cuda.Stream(device=local_rank, priority=-1)
                    comm.side_ctas = int(os.environ.get("UQB_MG_SIDE_CTAS", "2"))
                    exchange += "; on a side stream (%d CTAs per SM) next to the partition / sort of the neighbouring tables" % comm.side_ctas
            except Exception as e:                       # no peer mapping on this box: NCCL all-to-all
                comm.window = None
                exchange = "nccl all_to_all (peer window unavailable: %s)" % str(e).splitlines()[0][:120]
        else:
            exchange = "nccl all_to_all"

    parity = None
    if global_mode and not args.no_parity:
        parity = parity_check(ctx, comm, rank, world, host, multigpu, opts)
        if not parity["ok"]:
            if rank == 0:
                emit({"metric": "fastq_to_uq_encode_reads_per_s", "value": None, "n_gpus": world, "parity_check": parity,
                      "error": "sharded encode differs from the single-GPU encode"})
            dist.destroy_process_group()
            sys.exit(3)

    kept = []

    def one_step(keep=False):
        fq = ctx.adopt_fastq(dev)
        if global_mode:
            # ONE container from all ranks: global statistics, sample-sort unique (NCCL all-to-all), global order
            res, cfg = multigpu.encode_sharded(ctx, comm, fq, **opts)
            out_bytes = sum(a.nbytes for a, _, _ in res.slices.values())
            res.free()
        else:
            members, cfg = host.encode_device(ctx, fq, **opts)
            out_bytes = members.nbytes()
            if keep:
                kept.append(members)
            else:
                members.free()
        fq.free()
        return out_bytes, cfg

    for _ in range(args.warmup):
        out_bytes, cfg = one_step()
    if global_mode and os.environ.get("UQB_MG_TRACE") == "1" and rank == 0:
        print("trace (last warm-up step):", multigpu.trace_dump()[-40:], file=sys.stderr)
    ctx.sync()
    ctx.timing(True)
    ctx.timing_reset()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    launches0 = ctx.launches
    hc0 = list(comm.host_collectives) if global_mode else None
    ctx.span_begin()
    for i in range(args.steps):
        out_bytes, cfg = one_step(keep=bool(args.dump_outputs) and i == args.steps - 1)
    ms = ctx.span_end()
    barrier()
    clocks = sampler.stop() if sampler else None
    launches = ctx.launches - launches0
    host_coll = None
    if global_mode:
        host_coll = {"calls_per_step": (comm.host_collectives[0] - hc0[0]) / args.steps,
                     "ms_per_step_rank0": round((comm.host_collectives[1] - hc0[1]) * 1e3 / args.steps, 2),
                     "transport": "shared-memory board (one node)" if comm.board is not None else "gloo all_gather_object"}
    report = ctx.timing_report()
    ctx.timing(False)
    if kept:
        # before the decode and e2e legs, which need the HBM these members hold
        dump_outputs(args.dump_outputs, kept[0].download())
        kept[0].free()
    ms = max_over_ranks(ms)
    total_reads = sum_over_ranks(float(n))
    total_fbytes = sum_over_ranks(float(fbytes))
    total_out = sum_over_ranks(float(out_bytes))
    t = ms / 1e3 / args.steps
    value = total_reads / t

    # ---- roofline of the dominant kernel (rank 0's launches) ----
    peak, peak_src = peaks()
    kern = sorted(report.items(), key=lambda kv: -kv[1][1])
    kernel_ms = sum(v[1] for v in report.values())
    top_name, (top_cnt, top_ms, top_bytes) = kern[0]
    # prefer the heaviest kernel that carries an algorithmic byte count
    for name, (cnt, kms, kb) in kern:
        if kb > 0:
            top_name, top_cnt, top_ms, top_bytes = name, cnt, kms, kb
            break
    achieved = top_bytes / 1e9 / (top_ms / 1e3) if top_ms > 0 else 0.0
    roofline = {"bound": "hbm", "kernel": top_name, "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": None, "peak_source": peak_src,
                "launches_per_step": top_cnt / args.steps, "avg_launch_ms": round(top_ms / max(top_cnt, 1), 4),
                "share_of_step": round(top_ms / (ms * 1.0), 4), "algorithmic_bytes_per_launch": top_bytes / max(top_cnt, 1)}
    # DRAM traffic of the same kernel from the committed `ncu --set full` capture (same workload, per launch)
    try:
        with open(os.path.join(ROOT, "profiles", "r02_ncu_full_100m_summary.json")) as f:
            unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}

            def nbytes(txt):
                v, u = txt.split()
                return float(v) * unit[u]
            for rec in json.load(f):
                base = rec["kernel"].replace("void ", "").split("<")[0]        # the timer names template instances base_variant
                if (top_name.split("<")[0] == base or top_name.startswith(base + "_")) and n == 100_000_000:
                    measured = nbytes(rec["dram__bytes_read.sum"]) + nbytes(rec["dram__bytes_write.sum"])
                    # a kernel launched many times per step (radix passes: the three 100 M-row sorts and the small dictionary
                    # sorts) was captured at its full size; its DRAM / algorithmic ratio is applied to the average launch
                    captured_alg = {"k_radix_scatter_key": 24.0 * n}.get(top_name)
                    if captured_alg and top_cnt > args.steps:
                        roofline["traffic"] = measured / captured_alg * roofline["algorithmic_bytes_per_launch"]
                        roofline["traffic_note"] = ("captured launch: %d keys, %.3f GB of DRAM traffic for %.3f GB algorithmic; scaled to the "
                                                    "average of the %d launches per step" % (n, measured / 1e9, captured_alg / 1e9, top_cnt // args.steps))
                    else:
                        roofline["traffic"] = measured
                    roofline["traffic_source"] = "profiles/r02_ncu_full_100m_summary.json (dram__bytes_read.sum + dram__bytes_write.sum)"
                    break
    except Exception:
        pass
    a_enc = total_fbytes + total_out
    pipeline = {"algorithmic_bytes_per_step": a_enc, "achieved_GBps": round(a_enc / 1e9 / t, 1),
                "frac_of_peak": round(a_enc / 1e9 / t / (peak * world), 4),
                "kernel_time_share": round(kernel_ms / ms, 4)}
    top5 = [{"kernel": k, "launches": v[0], "ms": round(v[1], 3), "share": round(v[1] / ms, 4),
             "GBps": round(v[2] / 1e9 / (v[1] / 1e3), 1) if v[1] > 0 and v[2] else None} for k, v in kern[:8]]

    # ---- decode (SURVEY 8d), N = 1 only: three measurements, everything resident in HBM, text compared on the device ----
    decode = None
    if world == 1 and not args.no_decode:
        used, free, total = ctx.mem_info()
        if total - used > 2.8 * fbytes:             # the arena keeps what it mapped: room = total - bytes in use
            decode = decode_block(ctx, host, dev, n, fbytes, peak, args.steps)
        else:
            decode = {"value": None, "note": "skipped: needs %.0f GB of free HBM" % (2.6 * fbytes / 1e9)}

    # ---- end to end: host buffers, H2D + D2H inside the timed region ----
    e2e = None
    e2e_skip = None
    if not args.no_e2e:
        # the host copies are pinned: make sure every rank of this node can hold its input + outputs
        avail = 0
        try:
            with open("/proc/meminfo") as f:
                for ln in f:
                    if ln.startswith("MemAvailable:"):
                        avail = int(ln.split()[1]) * 1024
        except Exception:
            pass
        need = int((fbytes + out_bytes * 1.05) * 1.25)
        local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
        if avail and need * local_world > avail:
            e2e_skip = "skipped: %d ranks x %.0f GB of pinned host memory exceed the %.0f GB available" % (
                local_world, need / 1e9, avail / 1e9)
    if not args.no_e2e and e2e_skip is None:
        pin_in = ctx.pinned_empty(fbytes)
        ctx.check(ctx.lib.uqb_array_download(ctx.h, dev.h, pin_in.ptr, fbytes))
        dev.free()
        pin_out = ctx.pinned_empty(int(out_bytes * 1.05) + (1 << 20))

        def e2e_step():
            # H2D in chunks on the copy stream, overlapped with record splitting and the Pass-1 statistics;
            # every output array starts its D2H copy as soon as it is final
            cur = [0]

            def sink(name, nbytes):
                a = pin_out.array[cur[0]:cur[0] + nbytes]
                cur[0] += (nbytes + 63) & ~63
                return a
            if global_mode:
                # the global first QNAME line is read from rank 0's host buffer, so every rank can measure its
                # Pass-1 statistics against it while its own chunks are still streaming in
                line1 = bytes(pin_in.array[:min(int(fbytes), 4096)]).split(b"\n")[0]
                ref = comm.all_gather_object(line1)[0]
                fq = ctx.load_fastq_streamed(pin_in, ref=ref, rbase=0 if rank == 0 else 1)
                members, _ = multigpu.encode_sharded(ctx, comm, fq, sink=sink, **opts)
                members.download()
                nb = members.nbytes()
                members.free()
                fq.free()
                return nb
            fq = ctx.load_fastq_streamed(pin_in) if not args.e2e_serial else ctx.load_fastq(pin_in)
            if args.e2e_serial:
                members, _ = host.encode_device(ctx, fq, **opts)
                members.download(into=sink)
            else:
                members, _ = host.encode_device(ctx, fq, sink=sink, **opts)
                members.download()                      # waits for the copy stream
            nb = members.nbytes()
            members.free()
            fq.free()
            return nb
        e2e_step()
        ctx.sync()
        barrier()
        t0 = time.perf_counter()
        step_ms = []
        for _ in range(args.steps):
            ts = time.perf_counter()
            d2h = e2e_step()
            step_ms.append(round((time.perf_counter() - ts) * 1e3, 1))
        ctx.sync()
        barrier()
        te = max_over_ranks(time.perf_counter() - t0) / args.steps
        e2e = {"value": total_reads / te, "unit": "reads/s", "h2d_bytes_per_step": int(fbytes) * world,
               "d2h_bytes_per_step": int(d2h) * world, "ms_per_step": round(te * 1e3, 2), "ms_steps_rank0": step_ms,
               "overlap": "serial" if args.e2e_serial else "H2D chunks overlapped with split+Pass-1, D2H per output array as soon as final"}
        sample_src = pin_in
    else:
        sample_src = None
        if e2e_skip:
            e2e = {"value": None, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "note": e2e_skip}

    # ---- CPU baseline: the reference algorithm (oracle port) on a bounded sample, rank 0 at N=1 only ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import uq_literal as lit
        s_reads = args.cpu_sample
        if sample_src is not None:
            head = bytes(sample_src.array[:min(fbytes, s_reads * 420)])
        else:
            head = dev.download()[:s_reads * 420].tobytes()
        lines = head.split(b"\n")
        sample = b"\n".join(lines[:4 * s_reads]) + b"\n"
        t0 = time.perf_counter()
        lit.encode(sample, sort=SORT)
        dt = time.perf_counter() - t0
        cpu = {"value": round(s_reads / dt, 1), "unit": "reads/s", "cores": 1, "kind": "port",
               "sample": "first %d reads of the same FASTQ, full encode incl. --sort DNA (sort is over the sample only), %.1f s; "
                         "host has %d cores, the reference is single threaded" % (s_reads, dt, os.cpu_count())}

    if rank == 0:
        line = {
            "metric": "fastq_to_uq_encode_reads_per_s", "value": value, "unit": "reads/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
            "scaling": "strong" if (args.strong and world > 1) else "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "configs[1]: %d reads x %d bp per GPU, --sort DNA, keyed DNA/QUAL/QNAME tables, pattern 0.1 0.1"
                                   % (n, READ_LEN),
                       "reads_per_gpu": n, "read_len": READ_LEN, "fastq_bytes_per_gpu": int(fbytes),
                       "output_bytes_per_gpu": int(out_bytes), "genome": genome, "qual_pool": pool,
                       "l2": "inputs (%.1f GB) far larger than the 126 MB L2; no flush needed" % (fbytes / 1e9),
                       "bits": [cfg["bits_per_base"], cfg["bits_per_quality"]],
                       "sharding": ("contiguous read ranges per rank, ONE global container: merged statistics, sample-sort unique with "
                                    "NCCL all-to-all, global --sort order" if global_mode else
                                    "independent read ranges per rank, one container shard per rank (no data-path collective)")},
            "gb_per_s": round(total_fbytes / 1e9 / t, 2),
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline,
            "pipeline_roofline": pipeline, "kernels": top5, "decode": decode, "cpu_baseline": cpu,
        }
        if parity is not None:
            line["parity_check"] = parity
        if global_mode:
            line["config"]["row_exchange"] = exchange
            line["host_collectives"] = host_coll
        emit(line)
    if global_mode:
        comm.close()
    if dist is not None:
        dist.destroy_process_group()


def decode_block(ctx, host, dev, n, fbytes, peak, steps):
    """uQ -> FASTQ on the device.
      value / tables     packed DNA / QUAL tables and QNAME columns of the benched file (record order) -> text, compared
                         byte for byte with the input (the round-1 measurement)
      from_members       the members of a keyed container in layout 2.2 (--sort DNA --pattern 2.2 2.2): layouts undone,
                         keys widened and checked, unique rows gathered, text produced (uq.py:943-973 + 1002-1058)
      variable_length    configs[4]: 1 M reads of 1-20 kb, packed tables -> text, compared byte for byte with the input"""
    def timed(fn):
        fn().free()                                            # warm-up
        ctx.sync()
        ctx.span_begin()
        for _ in range(steps):
            fn().free()
        return ctx.span_end() / steps

    out = {}
    # ---- tables in record order ----
    fq = ctx.adopt_fastq(dev)
    st = {}
    dmembers, dcfg = host.encode_device(ctx, fq, sort="None", raw=["DNA", "QUAL", "QNAME"], stages=st)
    text = host.decode_device(ctx, st["dna"], st["qual"], st["cols"], dcfg)
    same = text.first_difference(dev) == -1
    text.free()
    dms = timed(lambda: host.decode_device(ctx, st["dna"], st["qual"], st["cols"], dcfg))
    tab_bytes = st["dna"].nbytes + st["qual"].nbytes + sum(c.nbytes for c in st["cols"])
    out.update({"value": n / (dms / 1e3), "unit": "reads/s", "ms_per_step": round(dms, 3),
                "gb_per_s_fastq": round(fbytes / 1e9 / (dms / 1e3), 2),
                "algorithmic_GBps": round((tab_bytes + fbytes) / 1e9 / (dms / 1e3), 1),
                "frac_of_peak": round((tab_bytes + fbytes) / 1e9 / (dms / 1e3) / peak, 4), "byte_exact": bool(same),
                "workload": "uQ -> FASTQ of the same %d reads: packed DNA / QUAL tables and QNAME columns resident in HBM -> "
                            "FASTQ text resident in HBM, compared byte for byte with the input on the device" % n})
    dmembers.free()
    fq.free()
    # ---- from the members of a keyed, transposed container ----
    fq = ctx.adopt_fastq(dev)
    km, kcfg = host.encode_device(ctx, fq, sort="DNA", pattern=["2.2", "2.2"])
    fq.free()
    text = host.decode_members_device(ctx, km, kcfg)
    size_ok = text.nbytes == fbytes
    text.free()
    kms = timed(lambda: host.decode_members_device(ctx, km, kcfg))
    mbytes = km.nbytes()
    out["from_members"] = {"ms_per_step": round(kms, 3), "value": n / (kms / 1e3), "unit": "reads/s",
                           "algorithmic_GBps": round((mbytes + fbytes) / 1e9 / (kms / 1e3), 1),
                           "frac_of_peak": round((mbytes + fbytes) / 1e9 / (kms / 1e3) / peak, 4), "text_bytes_ok": bool(size_ok),
                           "workload": "members of the keyed container of the same file (--sort DNA --pattern 2.2 2.2, %.1f GB): "
                                       "unlayout + key check + unique-row gather + text; record order = DNA order "
                                       "(round trip checked by tests/test_gpu_scale.py)" % (mbytes / 1e9)}
    km.free()
    # ---- configs[4]: variable-length long reads ----
    import numpy as np
    # the generator's table of 4096 log-spaced read lengths (same formula as the host generator of the tests)
    tab = np.clip(np.floor(1000 * np.power(20000.0 / 1000.0, np.arange(4096, dtype=np.float64) / 4096.0)).astype(np.int64), 1000, 20000)
    vn = 1_000_000
    vdev = ctx.synth("ont", vn, (1000, 20000), 1005, len_table=tab)
    fq = ctx.adopt_fastq(vdev)
    vst = {}
    vm, vcfg = host.encode_device(ctx, fq, sort="None", raw=["DNA", "QUAL", "QNAME"], stages=vst)
    text = host.decode_device(ctx, vst["dna"], vst["qual"], vst["cols"], vcfg)
    vsame = text.first_difference(vdev) == -1
    text.free()
    vms = timed(lambda: host.decode_device(ctx, vst["dna"], vst["qual"], vst["cols"], vcfg))
    # algorithmic bytes: the SIGNIFICANT part of the right-aligned rows (2 + 7 bits per base) + columns + text
    sig = (vcfg["bits_per_base"] + vcfg["bits_per_quality"]) / 8.0 * (vdev.nbytes / 2.0)
    vab = sig + sum(c.nbytes for c in vst["cols"]) + vdev.nbytes
    out["variable_length"] = {"ms_per_step": round(vms, 3), "value": vn / (vms / 1e3), "unit": "reads/s",
                              "gb_per_s_fastq": round(vdev.nbytes / 1e9 / (vms / 1e3), 2),
                              "algorithmic_GBps": round(vab / 1e9 / (vms / 1e3), 1), "frac_of_peak": round(vab / 1e9 / (vms / 1e3) / peak, 4),
                              "byte_exact": bool(vsame),
                              "workload": "configs[4]: %d reads of 1-20 kb (%.1f GB of FASTQ), tables %d + %d bytes per row "
                                          "(right aligned, significant bytes counted) -> text" % (vn, vdev.nbytes / 1e9, vst["dna"].width, vst["qual"].width)}
    vm.free(); fq.free(); vdev.free()
    return out


def parity_check(ctx, comm, rank, world, host, multigpu, opts, n_each=200_000):
    """The sharded path against the single-GPU path on a file small enough for rank 0 to encode alone: every member
    (dtype, shape, bytes) and the config of the global container must equal the single-GPU container, and the sharded
    decode of it must reproduce the single-GPU decode.  Runs with the bench's own options (--sort DNA, keyed)."""
    import numpy as np
    kw = dict(genome=n_each * world // 10, pool=max(1, n_each * world // 5))
    dev = ctx.synth("genome", n_each, READ_LEN, SEED + 1, first=rank * n_each, **kw)
    fq = ctx.adopt_fastq(dev)
    res, cfg = multigpu.encode_sharded(ctx, comm, fq, **opts)
    members = multigpu.assemble(comm, res)
    res.free(); fq.free(); dev.free()
    bad, k = [], 0
    if rank == 0:
        whole = ctx.synth("genome", n_each * world, READ_LEN, SEED + 1, first=0, **kw)
        wfq = ctx.adopt_fastq(whole)
        wm, wcfg = host.encode_device(ctx, wfq, **opts)
        want = wm.download()
        if sorted(want) != sorted(members):
            bad.append("member names")
        else:
            for name in want:
                a, b = members[name], np.asarray(want[name])
                k += 1
                if a.dtype != b.dtype or a.shape != b.shape or not np.array_equal(a, b):
                    bad.append(name)
        if json.loads(json.dumps(cfg, default=str)) != json.loads(json.dumps(wcfg, default=str)):
            bad.append("config.json")
        single_text = host.decode(want, wcfg, ctx=ctx).tobytes()
        wm.free(); wfq.free(); whole.free()
    members = comm.all_gather_object(members)[0]
    text, a, b = multigpu.decode_sharded(ctx, comm, members, cfg)
    texts = comm.all_gather_object(bytes(text))
    if rank == 0 and b"".join(texts) != single_text:
        bad.append("sharded decode")
    bad = comm.all_gather_object(bad)[0]
    return {"ranks": world, "reads": n_each * world, "members": k if rank == 0 else None, "decode": "sharded decode == single-GPU decode",
            "ok": not bad, "mismatches": bad}


def _ref_worker(job):
    """One host core: generate its own sample with the host generator, encode it with the oracle port."""
    idx, s_reads, steps = job
    from oracle import synth, uq_literal as lit
    fq = synth.make_fastq(kind="genome", n=s_reads, length=READ_LEN, seed=SEED, first=idx * s_reads,
                          genome=GENOME, pool=max(1, s_reads // 5))
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        lit.encode(fq, sort=SORT)
        times.append(time.perf_counter() - t0)
    return times


def run_reference(args):
    """The reference's own algorithm (py3 restatement of uq.py; the Python-2 original cannot run here) on the
    host cores: one independent process per core, each encoding its own bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    s_reads = args.ref_sample
    total_steps = args.warmup + args.steps
    with mp.Pool(cores) as pool:
        res = pool.map(_ref_worker, [(i, s_reads, total_steps) for i in range(cores)])
    per_step = [max(r[k] for r in res) for k in range(args.warmup, total_steps)]
    t = sum(per_step) / len(per_step)
    value = cores * s_reads / t
    line = {
        "impl": "reference", "metric": "fastq_to_uq_encode_reads_per_s", "value": value, "unit": "reads/s",
        "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(t * 1e3, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": "configs[1] shape: %d bp reads, --sort DNA, keyed tables; bounded sample of %d reads per core"
                               % (READ_LEN, s_reads)},
        "cpu_baseline": {"value": value, "unit": "reads/s", "cores": cores, "kind": "port",
                         "sample": "%d processes x %d reads each (reference algorithm is single threaded; one independent "
                                   "encode per core, sort over the sample only)" % (cores, s_reads)},
        "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=int(os.environ.get("UQ_BENCH_READS", "100000000")), help="reads per GPU")
    ap.add_argument("--cpu-sample", type=int, default=60000)
    ap.add_argument("--ref-sample", type=int, default=20000)
    ap.add_argument("--multi", default=os.environ.get("UQ_BENCH_MULTI", "global"), choices=["shards", "global"],
                    help="N>1: independent container shards per rank, or one global container (collectives on the data path)")
    ap.add_argument("--strong", action="store_true", help="N>1: --reads is the TOTAL number of reads (strong scaling) instead of reads per GPU")
    ap.add_argument("--no-p2p", action="store_true", help="N>1: row exchanges through NCCL all-to-all instead of direct stores into peer memory")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-decode", action="store_true")
    ap.add_argument("--e2e-serial", action="store_true", help="e2e without copy/compute overlap (diagnostics)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="N>1: skip the sharded-vs-single parity check before the timed loop")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the output arrays of the last timed step as DIR/<name>.npy "
                                                          "(float32 / float64, a seeded sample of each large array, < 64 MB)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
