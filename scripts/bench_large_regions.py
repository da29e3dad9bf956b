#!/usr/bin/env python
"""BASELINE.json configs[3] in the shape bench.py --workload configs3 uses (synth.config4: 100,000 samples = 200,000 haplotypes, a
record every ~4 bp, 32 regions, 50 PWMs on both strands), run two ways in the same process, the steps alternating:

  (a) one_block      the whole cohort as ONE block: most regions have more distinct haplotypes than the fan-out's shared-memory
                     count vector holds, so the fan-out keeps its count vectors in device memory (k_fanout<true>)
  (b) sample_blocks  five blocks of 20,000 samples (the fan-out in shared memory), rows_mode ALL_KEYS, merged on the host by
                     tfbs_merge_sample_blocks -- what bench.py --workload configs3 does

Both arms keep their blocks resident in HBM (tfbs_upload_block once, tfbs_run_resident per step).  A step ends with the grouped rows
on the host (tfbs_collect_grouped waits for the device) and, in arm (b), merged; it is timed with the host clock.  Per arm: ms per
step, ms_count (fan-out + row headers) and ms_total from tfbs_stats (summed over the blocks of a step), device memory the arm's
contexts hold (cudaMemGetInfo before / after, so other users of the GPU can blur it), device -> host bytes, and whether the two arms
give the same rows (keys, min and max).  The rows are only required to agree when no sequence-keyed overwrite happened in either arm
(tfbs_stats.n_dropped = 0): the winner of an overwrite is chosen per block.  The card's name and power limit are read in the same run.

  python scripts/bench_large_regions.py [--steps 10] [--min-seconds 0.5] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_identity():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                             text=True, timeout=60).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:  # the card's name still comes from the CUDA runtime
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % e}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--regions", type=int, default=32)
    ap.add_argument("--samples", type=int, default=100000)
    ap.add_argument("--block", type=int, default=20000, help="samples per sample block of arm (b)")
    ap.add_argument("--steps", type=int, default=10, help="at least this many timed steps per arm")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--min-seconds", type=float, default=0.5, help="and at least this much timed work per arm")
    ap.add_argument("--scratch-mb", type=int, default=65536, help="option scratch_mb of both arms (the one block's scratch estimate is "
                    "30.9 GB, more than the default 24 GB)")
    ap.add_argument("--out", default="", help="also write the JSON here")
    args = ap.parse_args()

    import numpy as np
    import torch
    from find_tfbs_b200 import binding, sharding, synth
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU fallback")
    torch.cuda.init()

    pats, blk = synth.config4(n_regions=args.regions, n_samples=args.samples)
    ps = binding.PatternSet(pats)
    S = blk.n_samples
    cuts = [(a, min(S, a + args.block)) for a in range(0, S, args.block)]
    parts_in = [sharding.sample_block(blk, a, b) for a, b in cuts]

    def context(mode, block):
        c = binding.Context(0)
        c.set_option("rows_width", 0)
        c.set_option("rows_mode", mode)
        c.set_option("scratch_mb", args.scratch_mb)
        c.set_patterns(ps)
        c.upload_block(block)
        return c

    def free_bytes():
        torch.cuda.synchronize()
        return torch.cuda.mem_get_info(0)[0]

    free0 = free_bytes()
    one = context(binding.ROWS_VARYING, blk)
    many = [context(binding.ROWS_ALL_KEYS, b) for b in parts_in]

    def step_one():
        one.run_resident()
        g = one.collect_grouped()
        st = one.stats()
        rows = {k: np.array(g[k]) for k in ("region", "inner", "pattern_id", "vmin", "vmax")}
        return rows, [st]

    def step_many():
        for c in many:
            c.run_resident()
        parts, sts = [], []
        for c in many:
            parts.append(binding.own_grouped(c.collect_grouped()))
            sts.append(c.stats())
        m = binding.merge_sample_blocks(parts, expand=False)
        return {k: m[k] for k in ("region", "inner", "pattern_id", "vmin", "vmax")}, sts

    arms = {"one_block": step_one, "sample_blocks": step_many}
    held = {}  # device memory an arm's contexts allocate while it warms up (scratch, results); the uploaded blocks are not counted
    last = {}
    for name, fn in arms.items():  # warm-up; the first run of a fresh context repeats until its capacities fit
        f = free_bytes()
        for _ in range(max(1, args.warmup)):
            last[name] = fn()
        held[name] = f - free_bytes()
    held_total = free0 - free_bytes()
    times = {name: [] for name in arms}
    t_start = time.perf_counter()
    while any(len(v) < args.steps or sum(v) < args.min_seconds for v in times.values()):
        for name, fn in arms.items():
            torch.cuda.synchronize()
            t = time.perf_counter()
            last[name] = fn()
            times[name].append(time.perf_counter() - t)
        if time.perf_counter() - t_start > 600:
            break

    out = {"what": "BASELINE.json configs[3] (synth.config4): %d samples x %d regions x 50 PWMs (both strands); (a) one block, (b) %d sample blocks "
                   "of <= %d merged by tfbs_merge_sample_blocks; resident blocks, steps alternating" % (S, blk.n_regions, len(cuts), args.block),
           "gpu": gpu_identity(), "arms": {}}
    for name in arms:
        rows, sts = last[name]
        tot = lambda k: sum(st[k] for st in sts)
        ts = np.array(times[name]) * 1e3
        out["arms"][name] = {"blocks": len(sts), "steps": len(ts), "ms_per_step": float(ts.mean()), "ms_per_step_min": float(ts.min()),
                             "ms_per_step_max": float(ts.max()), "ms_count": tot("ms_count"), "ms_total": tot("ms_total"),
                             "ms_count_share_of_total": tot("ms_count") / tot("ms_total") if tot("ms_total") else None,
                             "device_mb_held": held[name] / 2 ** 20, "d2h_bytes": int(tot("d2h_bytes")), "rows": int(len(rows["region"])),
                             "groups": int(tot("n_groups")), "n_dropped": int(tot("n_dropped")), "total_launches": int(tot("total_launches"))}
    out["device_mb_held_both_arms"] = held_total / 2 ** 20  # with the contexts and the uploaded blocks
    ra, rb = last["one_block"][0], last["sample_blocks"][0]
    same = len(ra["region"]) == len(rb["region"]) and all(np.array_equal(ra[k], rb[k]) for k in ra)
    dropped = out["arms"]["one_block"]["n_dropped"] + out["arms"]["sample_blocks"]["n_dropped"]
    out["rows_equal"] = bool(same)
    out["rows_equal_required"] = dropped == 0
    if dropped == 0 and not same:
        print(json.dumps(out))
        raise SystemExit("the two arms disagree although no overwrite happened")
    one.close()
    for c in many:
        c.close()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
