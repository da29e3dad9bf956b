#!/usr/bin/env python
"""bench.py -- find-tfbs hot path on B200: PWM cells/s (haplotype bp x PWM columns) on the north-star workload.

Workload (BASELINE.json configs[2]): ONE fixed synthetic block -- 2,504 samples (1000G-like) x 2 BED sets x 5,000 regions each
(4,873 merged regions) x 401 random PWMs on both strands, p = 1e-4 -- STRONG-scaled: the block is cut into contiguous region ranges
balanced by device work (find_tfbs_b200/sharding.py), one process + one context per GPU, no collective on the data path (regions are
independent, reference main.rs:395-429).  A step = one pass of the whole hot path (grouping, haplotype build, PWM scan on both
strands, per-haplotype counts, min/max row filter) over the whole block.

  value     nominal cells/s (every haplotype of every sample x every pattern), shards resident in HBM, device time (CUDA events)
  e2e       the same through tfbs_submit_block / tfbs_collect_grouped with HOST buffers: pinned inputs copied in, the grouped rows of
            every rank copied by its GPU straight into a shared-memory arena that rank 0 has mapped (tfbs_set_result_arena), rank 0
            reading every rank's rows inside the timed region; two blocks in flight per context
  roofline  the scan kernel against its lookup-add roof (DESIGN.md), timed with CUDA events on the library's kernel stream
  sustained the resident step repeated for >= 3 s, with the clocks seen meanwhile
  secondary BASELINE.json configs[1] (100 samples x 10k regions x 50 PWMs) on rank 0, N = 1 only: step, e2e, roofline, full-scan roofline
  cpu_baseline  the C++ oracle (a restatement of the reference: the Rust binary cannot be built here) on the host cores
  wall_s    chromosome wall time of the C++ driver (find-tfbs-b200) on the same cohort written as files, --devices 0..N-1 (rank 0)

`--impl reference` times the CPU restatement alone on the same workload.  Every context runs with option dual_stream (a twin context
on the same GPU: the blocks of consecutive steps alternate between two sets of streams and scratch and overlap on the device).
`--workload configs3` prints the line of BASELINE.json configs[3] instead: 200,000 haplotypes in SAMPLE BLOCKS, merged on the host by
tfbs_merge_sample_blocks (min != max over all samples after the gather), with `roofline_k1` for grouping + build.
`--dump-outputs DIR` writes the rows of the last timed step as .npy files (dump_outputs): the inputs are seeded, so two builds run
with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "pwm_cells_per_s"
UNIT = "cells/s"
SM_COUNT = 148
CELLS_PER_LDS64 = 6          # 3 packed patterns x 2 columns per 64-bit shared-memory read
LDS64_PER_CLK_PER_SM = 16    # 128 B/clk/SM of shared-memory bandwidth
DUMP_BYTES = 64 << 20        # --dump-outputs writes at most this much
DUMP_KEYS = ("region", "inner", "pattern_id", "vmin", "vmax")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="configs2", choices=["configs1", "configs2", "configs3"],
                    help="configs2 = BASELINE.json configs[2] (the north-star workload, default); configs1 = configs[1]")
    ap.add_argument("--c3-regions", type=int, default=32, help="configs3: merged regions of a step (the full config has 100k; regions are independent)")
    ap.add_argument("--c3-samples", type=int, default=100000, help="configs3: samples of the cohort (200k haplotypes)")
    ap.add_argument("--c3-block", type=int, default=20000, help="configs3: samples per sample block")
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the regions (debugging only)")
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="target duration of the CPU baseline sample")
    ap.add_argument("--ref-seconds-per-step", type=float, default=None, help="--impl reference: CPU seconds per step (default: 120 s over all steps, 2-30 s each)")
    ap.add_argument("--sustain-seconds", type=float, default=3.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the configs[1] object")
    ap.add_argument("--no-full-scan", action="store_true", help="skip the delta=0 pass that measures the scan kernel on the reference's full work")
    ap.add_argument("--no-driver", action="store_true", help="skip the wall time of the C++ driver on files")
    ap.add_argument("--option", action="append", default=[], help="library option key=value")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the rows of the last timed step to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200: the reference arm times a sample of the block sized by the clock")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d.get("hbm_gbs", 6650.0), "sm_max_mhz": d.get("sm_max_mhz", 1965.0), "source": "MEASURED_PEAKS.json"}
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": max(pw) if pw else None}


def workload(name, scale):
    from find_tfbs_b200 import synth
    if name == "configs2":
        pats, blk = synth.config3(scale=scale, seed=3)
        cfg = {"workload": "configs[2]: synthetic 2,504 samples (1000G-like allele-count spectrum) x 2 BED sets x %d regions each (%d merged regions) x 401 "
                           "random PWMs (L 7-25, both strands, p=1e-4); ONE fixed block, strong-scaled over the GPUs" % (int(5000 * scale), blk.n_regions),
               "regions": blk.n_regions, "samples": 2504, "pwms": 401, "patterns": 802}
    else:
        pats, blk = synth.config2(scale=scale, seed=2)
        cfg = {"workload": "configs[1]: synthetic 100 samples x %d DHS regions (200-2000 bp) x 50 random PWMs (L 8-30, both strands, p=1e-4); ONE fixed block"
                           % blk.n_regions, "regions": blk.n_regions, "samples": 100, "pwms": 50, "patterns": 100}
    cfg["sharding"] = "contiguous region ranges balanced by scan work, one context per GPU, no collective; rows land in rank 0's address space by DMA into shared memory"
    cfg["streams"] = "option dual_stream: the blocks of consecutive steps alternate between two contexts (streams + scratch) on the same GPU"
    cfg["l2"] = "inputs larger than L2 (carrier bits + reference windows + per-haplotype scratch of a step: hundreds of MB to GB)"
    return pats, blk, cfg


def cpu_reference_rate(pats, blk, seconds, threads):
    """Oracle (C++ restatement of the reference, multi-threaded like main.rs:333-382: workers pull chunks of merged regions from a
    shared queue) on a BOUNDED sample of the block, sized for about `seconds` of wall time: all samples, the first regions (at least
    one per thread), and -- when one region per thread with every pattern would already take longer, as on the 2,504-sample cohort
    (35 s) -- every k-th PWM of the list (both strands of a PWM stay together).  The reference's chunk is 50 regions (main.rs:378);
    a bounded sample uses min(50, regions / threads) so that every thread has work.  value = nominal cells of the sample / its time."""
    import parity_helpers as hp
    from find_tfbs_b200 import binding
    ids = sorted({p["pattern_id"] for p in pats})

    def subset(stride):
        keep = set(ids[::stride])
        return [p for p in pats if p["pattern_id"] in keep]

    n0 = min(blk.n_regions, max(threads, 8))
    stride = 1
    if len(ids) > 64:  # calibrate on a thin slice of the patterns: is one region per thread with all of them affordable?
        s0 = 32
        t = time.perf_counter()
        hp.run_oracle(binding.PatternSet(subset(s0)), blk.slice(0, n0), 0, False, threads, 1)
        est = (time.perf_counter() - t) * s0
        stride = max(1, min(len(ids), int(est / max(seconds, 1e-3) + 0.999)))
    sub = subset(stride)
    ps = binding.PatternSet(sub)
    t = time.perf_counter()
    o = hp.run_oracle(ps, blk.slice(0, n0), 0, False, threads, 1)
    dt = time.perf_counter() - t
    rate = o["nominal_cells"] / max(dt, 1e-9)
    n = int(min(blk.n_regions, max(n0, n0 * seconds / max(dt, 1e-6))))
    chunk = 1
    if n > n0 and stride == 1:
        chunk = max(1, min(50, n // threads))
        t = time.perf_counter()
        o = hp.run_oracle(ps, blk.slice(0, n), 0, False, threads, chunk)
        dt = time.perf_counter() - t
        rate = o["nominal_cells"] / max(dt, 1e-9)
    else:
        n = n0
    n_pwm = len({p["pattern_id"] for p in sub})
    return {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "seconds": dt, "executed_cells_per_s": o["executed_cells"] / max(dt, 1e-9),
            "regions": n, "chunk": chunk, "pwms": n_pwm,
            "sample": "first %d of %d merged regions of the block (%.1f %%), all %d samples, %s, %d threads pulling chunks of %d regions from a shared queue" %
                      (n, blk.n_regions, 100.0 * n / max(1, blk.n_regions), blk.n_samples,
                       "all patterns" if stride == 1 else "every %d-th PWM of the list (%d of %d, both strands)" % (stride, n_pwm, len(ids)), threads, chunk)}


def measured_traffic(workload, scale):
    """DRAM bytes of the k_scan launches of one step, from the committed `ncu --set full` capture of this workload at full scale
    (profiles/k_scan_traffic.json; not a live number).  None for any other workload or scale."""
    p = os.path.join(ROOT, "profiles", "k_scan_traffic.json")
    if scale != 1.0 or not os.path.exists(p):
        return None, None
    t = json.load(open(p)).get(workload)
    if not t:
        return None, None
    return t["dram_bytes_per_step"], "profiles/k_scan_traffic.json: " + t["source"]


def roofline_object(st, scan_ms, clocks, pk, traffic=None, traffic_source=None):
    scan_s = scan_ms * 1e-3
    achieved = st["evaluated_cells"] / scan_s
    f_max = pk["sm_max_mhz"] * 1e6
    sm_count = st["sm_count"] or SM_COUNT
    roof = sm_count * LDS64_PER_CLK_PER_SM * CELLS_PER_LDS64 * f_max
    f_obs = ((clocks or {}).get("sm_mhz") or pk["sm_max_mhz"]) * 1e6
    sb = st["scan_input_bytes"]
    return {"bound": "lookup-add (shared-memory table bandwidth; not hbm, not tensor: see DESIGN.md)", "kernel": "k_scan",
            "achieved": achieved / 1e12, "peak": roof / 1e12, "unit": "Tcell/s", "frac": achieved / roof,
            "peak_basis": "%d SMs x 128 B/clk shared memory = 16 LDS.64/clk/SM x 6 cells per LDS.64 (3 packed patterns x 2 columns) at sm_max_mhz from %s" % (sm_count, pk["source"]),
            "frac_at_observed_clock": achieved / (roof * f_obs / f_max), "observed_sm_mhz": (clocks or {}).get("sm_mhz"),
            "frac_of_one_lookup_per_cell_roof": achieved / (sm_count * 32 * f_max), "frac_of_int32_issue_roof": achieved / (sm_count * 128 * f_max),
            "ms_per_step": scan_ms, "launches_per_step": st["scan_launches"], "cells_per_step": st["evaluated_cells"],
            "traffic": traffic, "traffic_source": traffic_source,
            # the same launches seen from HBM: algorithmic bytes (12 B per 32 packed bases of every scored entry, once per pattern chunk,
            # + the tables once per CTA) over the same CUDA-event time: orders of magnitude under the copy bandwidth, i.e. not the bound
            "hbm": {"achieved_gbs": sb / scan_s / 1e9, "peak_gbs": pk["hbm_gbs"], "frac": sb / scan_s / 1e9 / pk["hbm_gbs"],
                    "algorithmic_bytes_per_step": sb, "bytes_per_cell": sb / max(1, st["evaluated_cells"])}}


def main():
    args = parse_args()
    # stdout carries exactly one JSON line: anything libraries print there (e.g. the NCCL version banner) goes to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(obj), flush=True)
        os.dup2(2, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    from find_tfbs_b200 import binding, sharding

    if args.impl == "reference":
        if rank != 0:
            return
        pats, blk, config = workload(args.workload, args.scale)
        ps = binding.PatternSet(pats)
        threads = os.cpu_count() or 1
        per_step = args.ref_seconds_per_step or max(2.0, min(30.0, 120.0 / max(1, args.steps + args.warmup)))
        vals = []
        info = None
        for i in range(args.warmup + args.steps):
            info = cpu_reference_rate(pats, blk, per_step, threads)
            if i >= args.warmup:
                vals.append((info["value"], info["seconds"]))
        v = sum(x[0] for x in vals) / max(1, len(vals))
        ms = 1000.0 * sum(x[1] for x in vals) / max(1, len(vals))
        info["value"] = v
        out = {"metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
               "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": config,
               "impl": "reference", "cpu_baseline": info,
               "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
               "note": "CPU restatement (oracle/) of the reference algorithm on all host cores; each step is a bounded sample of the workload, value = nominal cells of "
                       "the sample / its wall time; the Rust reference cannot be compiled in this image (no cargo/rustc)"}
        emit(out)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=600))

    def options(ctx):
        for kv in args.option:
            k, v = kv.split("=")
            ctx.set_option(k, int(v))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        if world == 1:
            return x
        t = torch.tensor([float(x)], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def total(x):
        if world == 1:
            return x
        t = torch.tensor([float(x)], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def pipelined(ctx, start, collect, steps):
        """`steps` blocks with two in flight: the next one is enqueued before the previous one is collected.  Returns what the last
        collect returned."""
        start()
        for _ in range(steps - 1):
            start()
            collect()
        return collect()

    def timed(ctx, stream, fn):
        """fn() bracketed by barrier + synchronize on both sides; device time from CUDA events on the library's kernel stream (they are
        reached when everything before them has run, the host-side waits of fn included); max over ranks."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        barrier()
        return allmax(e0.elapsed_time(e1))

    if args.workload == "configs3":
        if world != 1:
            raise SystemExit("--workload configs3 runs its sample blocks on one GPU (tests/test_multi_gpu.py covers two)")
        emit(configs3_line(args, binding, sharding, local_rank, ClockSampler, peaks()))
        return

    pats, blk, config = workload(args.workload, args.scale)
    lmax = max(p["weights"].shape[0] for p in pats)
    shard, r0, i0 = sharding.shard_block(blk, world, rank, lmax=lmax, compact=True)
    config["regions_this_rank"] = shard.n_regions
    ps = binding.PatternSet(pats)
    ctx = binding.Context(local_rank)
    ctx.set_option("rows_width", 0)
    ctx.set_option("dual_stream", 1)  # consecutive blocks run on two streams of the same GPU (a twin context): their kernels overlap
    options(ctx)
    ctx.set_patterns(ps)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local_rank))

    # ---- resident path: the shard in HBM, grouped rows collected (they stay on this rank) ----
    ctx.upload_block(shard)
    run, coll = ctx.run_resident, lambda: ctx.collect_grouped()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # the first two blocks size the scratch (each may be repeated once or twice); the third is the first one enqueued with the
    # capacities the device asked for (new shared-memory sizes, buffers): steady state starts with the fourth
    pipelined(ctx, run, coll, max(4, args.warmup))
    last = []
    ms_total = timed(ctx, stream, lambda: last.append(pipelined(ctx, run, coll, args.steps)))
    if args.dump_outputs:  # before the next collect reuses the buffers the rows point into
        dump_outputs(args.dump_outputs, {"rank%d_" % rank if world > 1 else "": last[0]}, DUMP_BYTES // world)
    st = ctx.stats()
    launches = st["total_launches"] * args.steps
    ms_step = ms_total / args.steps
    nominal = total(st["nominal_cells"])
    executed = total(st["executed_cells"])
    evaluated = total(st["evaluated_cells"])
    rows_total = total(st["n_rows"])
    value = nominal / (ms_step * 1e-3)
    # scan kernel time per step of this rank: CUDA events around the k_scan launches (tfbs_stats.ms_scan_kernel), averaged over a few steps
    scan_ms = []
    for _ in range(5):
        ctx.run_resident()
        ctx.collect_grouped()
        scan_ms.append(ctx.stats()["ms_scan_kernel"])
    scan_ms = sum(scan_ms) / len(scan_ms)
    stages = {k: ctx.stats()[k] for k in ("ms_group", "ms_build", "ms_scan", "ms_scan_kernel", "ms_count", "ms_total")}

    # ---- sustained: the same resident step for >= sustain-seconds, clocks sampled meanwhile ----
    sustained = None
    if args.sustain_seconds > 0:
        n_sus = max(args.steps, int(args.sustain_seconds * 1000.0 / max(ms_step, 1e-3)) + 1)
        ms_sus = timed(ctx, stream, lambda: pipelined(ctx, run, coll, n_sus))
        sustained = {"steps": n_sus, "seconds": ms_sus * 1e-3, "ms_per_step": ms_sus / n_sus, "value": nominal / (ms_sus / n_sus * 1e-3), "unit": UNIT}
    clocks = sampler.stop() if rank == 0 else None
    if sustained is not None and clocks is not None:
        sustained["clocks"] = clocks

    # ---- end to end: pinned host buffers in, grouped rows out into the shared-memory arena rank 0 maps ----
    shard.pin()
    ctx.submit_block(shard)
    probe = ctx.collect_grouped()
    tag = "%s_%d" % (os.environ.get("MASTER_PORT", "0"), os.getppid() if world > 1 else os.getpid())
    arena = sharding.SharedArena(tag, rank, nbytes=2 * (int(probe["bytes"] * 1.3) + (1 << 20)), create=True)
    ctx.set_result_arena(arena.buf)
    pipelined(ctx, lambda: ctx.submit_block(shard), coll, 4)  # every slot of both twins has received a block from host memory once
    barrier()
    others = [sharding.SharedArena(tag, k) for k in range(world)] if rank == 0 else []
    gathered = {}

    def e2e_steps():
        pipelined(ctx, lambda: ctx.submit_block(shard), coll, args.steps)
        if world > 1:
            dist.barrier()  # every rank's last block has landed in its arena
        if rank == 0:  # the gathering rank reads the rows of every GPU where the DMA put them: no copy, no collective
            n_rows, n_bytes, check = 0, 0, 0
            for a in others:
                for half in (0, 1):
                    g = binding.read_arena(a.buf, half)
                    if g is None:
                        continue
                    n_bytes += g["bytes"]
                    if half == (args.steps - 1) % 2:  # the half the last block went to
                        n_rows += g["n_rows"]
                        check ^= int(np.bitwise_xor.reduce(g["vmax"])) if g["n_rows"] else 0
            gathered.update({"rows_last_step": int(n_rows), "arena_bytes": int(n_bytes), "vmax_xor": check})

    ms_e2e = timed(ctx, stream, e2e_steps) / args.steps
    st2 = ctx.stats()
    e2e = {"value": nominal / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(total(st2["h2d_bytes"])),
           "d2h_bytes_per_step": int(total(st2["d2h_bytes"])), "ms_per_step": ms_e2e, "blocks_in_flight": 2,
           "rows": "grouped (one count per distinct haplotype of the region + the haplotype -> group map per region), copied by each GPU into a /dev/shm arena mapped by rank 0",
           "gathered_on_rank0": gathered if rank == 0 else None}
    if rank == 0:
        assert gathered.get("rows_last_step") == int(rows_total), (gathered, rows_total)
    ctx.set_result_arena(None)
    for a in others:
        a.close()
    barrier()
    arena.close()

    # the same through the dense (left, right) rows of the reference's count_matches_by_sample, one block at a time (N = 1 only)
    e2e_dense = None
    if world == 1:
        def dense_steps():
            for _ in range(max(2, args.steps // 4)):
                ctx.submit_block(shard)
                ctx.collect(copy=False)
        dense_steps()
        ms_d = timed(ctx, stream, dense_steps) / max(2, args.steps // 4)
        e2e_dense = {"value": nominal / (ms_d * 1e-3), "unit": UNIT, "ms_per_step": ms_d, "d2h_bytes_per_step": int(ctx.stats()["d2h_bytes"]),
                     "rows": "dense u8/u16/u32 (left, right) per sample, expanded on the device"}
    shard.unpin()

    # ---- full scan (delta scoring off): the scan kernel doing the reference's own work, for its roofline ----
    pk = peaks()
    full_scan = None
    if rank == 0 and not args.no_full_scan and args.workload == "configs1":
        full_scan = full_scan_roofline(ctx, shard, pk, clocks)

    if world > 1:  # the collective part is over: rank 0 goes on alone (driver wall time on all GPUs), the others release theirs
        dist.barrier()
        dist.destroy_process_group()
        if rank != 0:
            ctx.close()
            return

    roofline = roofline_object(st, scan_ms, clocks, pk, *(measured_traffic(args.workload, args.scale) if world == 1 else (None, None)))
    if full_scan:
        roofline["full_scan"] = full_scan
    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": config,
           "executed_cells_per_s": executed / (ms_step * 1e-3), "nominal_cells_per_step": nominal, "executed_cells_per_step": executed,
           "evaluated_cells_per_step": evaluated, "rows_per_step": rows_total,
           "cells": "nominal = every haplotype of every sample x every pattern; executed = distinct haplotypes only (what the reference scans); "
                    "evaluated = what k_scan scored (a patched haplotype is scored only where a window touches one of its records)",
           "rank0": {"stages_ms": stages, "groups": st["n_groups"], "hits": st["n_hits"], "rows": st["n_rows"], "scan_items": st["n_scan_items"],
                     "groups_dropped": st["n_dropped"], "haplotypes_truncated": st["n_truncated"], "launches_per_step": st["total_launches"],
                     "fanout_count_vectors": st["reserved"]},
           "roofline": roofline, "e2e": e2e, "e2e_dense_rows": e2e_dense, "sustained": sustained, "gpu_launches": launches, "clocks": clocks}

    ctx.close()
    if world == 1 and not args.no_secondary and args.workload == "configs2":
        try:
            out["secondary"] = secondary_configs1(args, binding, sharding, local_rank, pk)
        except Exception as exc:  # never let a secondary measurement break the contract line
            out["secondary"] = {"skipped": str(exc)[:300]}
    if not args.no_driver:
        try:
            out["wall_s"] = driver_wall_time(args, world, pats, blk)
        except Exception as exc:
            out["wall_s"] = {"skipped": str(exc)[:300]}
    if not args.no_cpu_baseline and world == 1:
        out["cpu_baseline"] = cpu_reference_rate(pats, blk, args.cpu_seconds, os.cpu_count() or 1)
    emit(out)


def full_scan_roofline(ctx, blk, pk, clocks):
    """The same block with every distinct haplotype scored in full (what the reference does): the scan kernel's own roofline."""
    ctx.set_option("delta", 0)
    ctx.upload_block(blk)
    ms = []
    for _ in range(3):
        ctx.run_resident()
        ctx.collect(copy=False)
        ms.append(ctx.stats()["ms_scan_kernel"])
    fst = ctx.stats()
    ctx.set_option("delta", 1)
    f_max = pk["sm_max_mhz"] * 1e6
    roof = (fst["sm_count"] or SM_COUNT) * LDS64_PER_CLK_PER_SM * CELLS_PER_LDS64 * f_max
    s = sum(ms[1:]) / len(ms[1:]) * 1e-3
    return {"note": "same block, delta scoring off (every distinct haplotype scored in full, like the reference)",
            "cells_per_step": fst["evaluated_cells"], "ms_per_step": s * 1e3, "achieved": fst["evaluated_cells"] / s / 1e12,
            "frac": fst["evaluated_cells"] / s / roof}


def secondary_configs1(args, binding, sharding, device, pk):
    """BASELINE.json configs[1] on one GPU: the workload of round 1's headline, kept for continuity."""
    import torch
    pats, blk, config = workload("configs1", args.scale)
    ps = binding.PatternSet(pats)
    ctx = binding.Context(device)
    ctx.set_option("rows_width", 0)
    ctx.set_option("dual_stream", 1)
    for kv in args.option:
        k, v = kv.split("=")
        ctx.set_option(k, int(v))
    ctx.set_patterns(ps)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", device))
    steps = max(20, args.steps)

    def timed(fn):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def pipelined(start, n):
        start()
        for _ in range(n - 1):
            start()
            ctx.collect_grouped()
        ctx.collect_grouped()

    ctx.upload_block(blk)
    pipelined(ctx.run_resident, 6)
    ms_step = timed(lambda: pipelined(ctx.run_resident, steps)) / steps
    st = ctx.stats()
    scan_ms = []
    for _ in range(5):
        ctx.run_resident()
        ctx.collect_grouped()
        scan_ms.append(ctx.stats()["ms_scan_kernel"])
    stages = {k: ctx.stats()[k] for k in ("ms_group", "ms_build", "ms_scan", "ms_scan_kernel", "ms_count", "ms_total")}
    blk.pin()
    pipelined(lambda: ctx.submit_block(blk), 4)
    ms_e2e = timed(lambda: pipelined(lambda: ctx.submit_block(blk), steps)) / steps
    st2 = ctx.stats()
    blk.unpin()
    roof = roofline_object(st, sum(scan_ms) / len(scan_ms), None, pk, *measured_traffic("configs1", args.scale))
    if not args.no_full_scan:
        roof["full_scan"] = full_scan_roofline(ctx, blk, pk, None)
    ctx.close()
    return {"config": config, "value": st["nominal_cells"] / (ms_step * 1e-3), "unit": UNIT, "ms_per_step": ms_step, "steps": steps,
            "e2e": {"value": st["nominal_cells"] / (ms_e2e * 1e-3), "ms_per_step": ms_e2e, "h2d_bytes_per_step": st2["h2d_bytes"], "d2h_bytes_per_step": st2["d2h_bytes"]},
            "stages_ms": stages, "evaluated_cells_per_step": st["evaluated_cells"], "executed_cells_per_step": st["executed_cells"],
            "rows_per_step": st["n_rows"], "launches_per_step": st["total_launches"], "roofline": roof}


def configs3_line(args, binding, sharding, device, ClockSampler, pk):
    """BASELINE.json configs[3] (biobank scale, sample-sharded): 200,000 haplotypes, a record every ~4 bp, 50 PWMs, a bounded number
    of the 100k regions per step.  The cohort is cut into SAMPLE BLOCKS (what a region's fan-out holds in shared memory bounds the
    distinct haplotypes per block); every block is run with rows_mode = ALL_KEYS and the min != max filter of main.rs:450-458 is
    applied after the gather by tfbs_merge_sample_blocks.  `value`: every block resident in HBM (one context each); `e2e`: one
    context, the blocks submitted from pinned host memory two in flight, grouped rows copied out and merged on the host.
    `roofline_k1` is SURVEY 8(d)'s "K1 / config 4" figure: algorithmic bytes of grouping + build over their device time."""
    import torch
    from find_tfbs_b200 import synth
    pats, blk = synth.config4(n_regions=args.c3_regions, n_samples=args.c3_samples)
    S = blk.n_samples
    cuts = [(a, min(S, a + args.c3_block)) for a in range(0, S, args.c3_block)]
    config = {"workload": "configs[3]: synthetic %d samples (%d haplotypes, a record every ~4 bp, 1/k allele-count spectrum, uniform carriers) x %d of the "
                          "100k regions (200-2000 bp) x 50 random PWMs (L 8-30, both strands, p=1e-4), in %d sample blocks of <= %d samples"
                          % (S, 2 * S, blk.n_regions, len(cuts), args.c3_block),
              "regions": blk.n_regions, "samples": S, "pwms": 50, "patterns": len(pats), "sample_blocks": len(cuts),
              "sharding": "sample blocks (counts are per sample; min != max over all samples after the gather, tfbs_merge_sample_blocks)",
              "l2": "inputs larger than L2 (carrier bits of a block: tens of MB; per-haplotype scratch: GBs)"}
    ps = binding.PatternSet(pats)
    blocks = [sharding.sample_block(blk, a, b) for a, b in cuts]

    def context():
        c = binding.Context(device)
        c.set_option("rows_width", 0)
        c.set_option("rows_mode", binding.ROWS_ALL_KEYS)
        for kv in args.option:
            k, v = kv.split("=")
            c.set_option(k, int(v))
        c.set_patterns(ps)
        return c

    def timed(stream, fn):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        torch.cuda.synchronize()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    # ---- resident: one context per sample block, its block in HBM ----
    ctxs = [context() for _ in blocks]
    for c, b in zip(ctxs, blocks):
        c.upload_block(b)
    stream = torch.cuda.ExternalStream(ctxs[0].stream(), device=torch.device("cuda", device))

    def step():
        for c in ctxs:
            c.run_resident()
        return [c.collect_grouped() for c in ctxs]

    sampler = ClockSampler(device)
    sampler.start()
    for _ in range(max(3, args.warmup)):
        step()
    last = []
    ms_step = timed(stream, lambda: last.append([step() for _ in range(args.steps)][-1])) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"block%d_" % i: g for i, g in enumerate(last[0])}, DUMP_BYTES)
    clocks = sampler.stop()
    sts = [c.stats() for c in ctxs]
    tot = lambda k: sum(st[k] for st in sts)
    nominal, executed, evaluated = tot("nominal_cells"), tot("executed_cells"), tot("evaluated_cells")
    stages = {k: tot(k) for k in ("ms_group", "ms_build", "ms_scan", "ms_scan_kernel", "ms_count", "ms_total")}
    st_sum = dict(sts[0])
    for k in ("evaluated_cells", "scan_input_bytes", "scan_launches", "total_launches"):
        st_sum[k] = tot(k)
    roofline = roofline_object(st_sum, stages["ms_scan_kernel"], clocks, pk)
    # K1 roof (HBM): what grouping + build must read -- the carrier bits of every in-window record, the records, the windows
    H = 2 * S
    k1_bytes = int(len(blk.variants) * (H / 8 + 32) + len(blk.ref_bases))
    k1_s = (stages["ms_group"] + stages["ms_build"]) * 1e-3
    roofline_k1 = {"bound": "hbm", "kernels": "K0 grouping + K1 build (k_signatures .. k_redirect)", "achieved": k1_bytes / k1_s / 1e9, "peak": pk["hbm_gbs"],
                   "unit": "GB/s", "frac": k1_bytes / k1_s / 1e9 / pk["hbm_gbs"], "algorithmic_bytes_per_step": k1_bytes,
                   "ms_per_step": k1_s * 1e3, "traffic": None,
                   "basis": "carrier bits V x H / 8 + 32 B per record + the reference windows, summed over the regions (SURVEY 8d); sequences are never "
                            "materialised (segments + 3 bits per scored base instead)"}
    for c in ctxs:
        c.close()

    # ---- end to end: one context, blocks from pinned host memory, two in flight; rows copied out; merge on the host ----
    ctx = context()
    blocks[0].pin()  # the sample blocks share every array but the carrier bits
    for b in blocks[1:]:
        if binding.lib().tfbs_host_register(b.carriers.ctypes.data, b.carriers.nbytes) != 0:
            raise SystemExit("cudaHostRegister failed")
    merged_info = {}

    def e2e_step():
        parts, d2h, h2d = [], 0, 0
        ctx.submit_block(blocks[0])
        for i in range(len(blocks)):
            if i + 1 < len(blocks):
                ctx.submit_block(blocks[i + 1])
            g = ctx.collect_grouped()
            d2h += ctx.stats()["d2h_bytes"]
            h2d += ctx.stats()["h2d_bytes"]
            parts.append(binding.own_grouped(g))
        m = binding.merge_sample_blocks(parts, expand=False)
        merged_info.update({"rows_all_keys": int(sum(p["n_rows"] for p in parts)), "rows_kept": int(len(m["region"])), "d2h": int(d2h), "h2d": int(h2d),
                            "vmax_xor": int(np_xor(m["vmax"]))})

    e2e_step()
    e2e_step()
    ms_e2e = timed(stream_of(torch, ctx, device), lambda: [e2e_step() for _ in range(args.steps)]) / args.steps
    launches = ctx.stats()["total_launches"]
    blocks[0].unpin()
    for b in blocks[1:]:
        binding.lib().tfbs_host_unregister(b.carriers.ctypes.data)
    ctx.close()
    out = {"metric": METRIC, "value": nominal / (ms_step * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup),
           "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
           "config": config, "executed_cells_per_s": executed / (ms_step * 1e-3), "nominal_cells_per_step": nominal,
           "executed_cells_per_step": executed, "evaluated_cells_per_step": evaluated, "rows_per_step": merged_info["rows_kept"],
           "stages_ms_summed_over_blocks": stages, "groups": tot("n_groups"), "hits": tot("n_hits"), "haplotypes_truncated": tot("n_truncated"),
           "groups_dropped": tot("n_dropped"), "roofline": roofline, "roofline_k1": roofline_k1,
           "e2e": {"value": nominal / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": merged_info["h2d"], "d2h_bytes_per_step": merged_info["d2h"],
                   "ms_per_step": ms_e2e, "blocks_in_flight": 2, "rows_all_keys": merged_info["rows_all_keys"], "rows_kept": merged_info["rows_kept"],
                   "vmax_xor": merged_info["vmax_xor"],
                   "rows": "grouped, ALL_KEYS per sample block; merged on the host by tfbs_merge_sample_blocks (inside the timed region)"},
           "gpu_launches": int(tot("total_launches")) * args.steps, "launches_per_block": launches, "clocks": clocks}
    if not args.no_cpu_baseline:
        small = sharding.sample_block(blk, 0, min(S, 2048))
        out["cpu_baseline"] = cpu_reference_rate(pats, small, args.cpu_seconds, os.cpu_count() or 1)
        out["cpu_baseline"]["sample"] = "first %d samples of the cohort; " % small.n_samples + out["cpu_baseline"]["sample"]
    return out


def dump_outputs(out_dir, parts, budget):
    """--dump-outputs: the rows the timed path handed its caller in its last step, as .npy files by which two builds can be compared.
    `parts` maps a file-name prefix to the grouped rows of one context (collect_grouped).  Per part, in the library's row order
    (deterministic, include/tfbs.h): DUMP_KEYS of the rows and `n_groups` of the regions as float64, and the per-sample counts
    `left` / `right` as float32 (exact: a count is bounded by the window length) for the rows listed in `dense_rows`.  The group
    labels of the grouped form are not results, so its packed arrays are written decoded (tfbs_expand_rows) rather than as they
    are.  Whatever exceeds the part's share of `budget` is a fixed, seeded sample of the rows."""
    import ctypes as C
    import numpy as np
    from find_tfbs_b200 import binding
    os.makedirs(out_dir, exist_ok=True)
    share = budget // max(1, len(parts)) - (1 << 12)  # room for the .npy headers

    def pick(n, k, rng):
        return np.arange(n) if k >= n else np.sort(rng.choice(n, max(0, k), replace=False))

    for prefix, g in parts.items():
        rng = np.random.default_rng(0)
        n, S = int(g["n_rows"]), int(g["n_samples"])
        out = {"n_groups": np.asarray(g["n_groups"], dtype=np.float64)}
        rows = pick(n, (share // 2 - out["n_groups"].nbytes) // (8 * (len(DUMP_KEYS) + 1)), rng)
        out["rows"] = rows.astype(np.float64)
        for k in DUMP_KEYS:
            out[k] = np.asarray(g[k], dtype=np.float64)[rows]
        dense = rows[pick(len(rows), (share // 2) // (8 * max(1, S) + 8), rng)]
        left, right = np.zeros((len(dense), S), np.uint32), np.zeros((len(dense), S), np.uint32)
        for j, r in enumerate(dense):
            rc = binding.lib().tfbs_expand_rows(C.byref(g["_c"]), int(r), 1, left[j].ctypes.data_as(C.POINTER(C.c_uint32)),
                                                right[j].ctypes.data_as(C.POINTER(C.c_uint32)))
            if rc != binding.TFBS_OK:
                raise binding.TfbsError(rc, "tfbs_expand_rows failed")
        out.update({"dense_rows": dense.astype(np.float64), "left": left.astype(np.float32), "right": right.astype(np.float32)})
        for k, a in out.items():
            np.save(os.path.join(out_dir, prefix + k + ".npy"), a)


def np_xor(a):
    import numpy as np
    return np.bitwise_xor.reduce(a) if len(a) else 0


def stream_of(torch, ctx, device):
    return torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", device))


def driver_wall_time(args, world, pats, blk):
    """Chromosome wall time: the C++ driver (the reference's command line on top of the library) on the cohort written as files
    (BCF + CSI, FASTA + .fai, two BED files, PWM + threshold files), one context per GPU (--devices 0..N-1).  The file set is read
    from scratch_data/ when scripts/make_cohort_files.py has written it there; otherwise it is written into a temporary directory
    first (about half a minute for configs[2], not timed)."""
    name = "cfg2" if args.workload == "configs2" else "cfg1"
    d = os.path.join(ROOT, "scratch_data", name if args.scale == 1.0 else "%s_%g" % (name, args.scale))
    argfile = os.path.join(d, "args.txt")
    exe = os.path.join(ROOT, "find_tfbs_b200", "find-tfbs-b200")
    if not os.path.exists(exe):
        return {"skipped": "no driver binary at %s" % exe}
    with tempfile.TemporaryDirectory(prefix="tfbs_bench_") as tmp:
        if os.path.exists(argfile):
            cli = open(argfile).read().split()
            cli = [a if not a.startswith("scratch_data/") else os.path.join(ROOT, a) for a in cli]
        else:
            sys.path.insert(0, os.path.join(ROOT, "scripts"))
            import make_cohort_files
            cli = make_cohort_files.write_file_set(pats, blk, tmp, tmp)
        outp = os.path.join(tmp, "out.vcf.gz")
        threads = os.cpu_count() or 8
        cmd = [exe] + cli + ["--output", outp, "--threads", str(threads), "--devices", ",".join(str(k) for k in range(world))]
        t = time.perf_counter()
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1500)
        dt = time.perf_counter() - t
        tail = [ln for ln in r.stdout.strip().split("\n")[-4:]]
        size = os.path.getsize(outp) if os.path.exists(outp) else 0
    if r.returncode != 0:
        return {"skipped": "driver failed: " + " | ".join(tail)[-300:]}
    return {"value": dt, "unit": "s", "devices": world, "host_threads": threads, "output_bytes": size, "command": "find-tfbs-b200 <file set of the same cohort> --devices 0..N-1",
            "phases": tail}


if __name__ == "__main__":
    main()
