#!/usr/bin/env python
"""What option "region_tables" changes on the BASELINE.json configs[2] block (synth.config3: 2,504 samples, two BED sets, 401 PWMs on
both strands), the shape bench.py measures.  Two contexts in one process, option 0 (K0 through the block-wide tables: k_signatures,
k_group_insert, k_group_lookup, k_group_rank, k_seq_init) and 1 (k_group_region, k_seq_init_groups), each with the block resident in
HBM (tfbs_upload_block once, tfbs_run_resident per step); the steps alternate between them.  A step ends with the grouped rows on the
host (tfbs_collect_grouped) and is timed with the host clock.

Reported per arm: ms per step (median, mean, min), the stage times of tfbs_stats (ms_group = K0 up to the scan of the group counts,
ms_build, ms_scan, ms_count, ms_total; CUDA events of the last step), and the device time per kernel of one step from a separate
torch.profiler run.  The grouped rows of the two arms are compared.  The card's name and power limit are read in the same run.

  python scripts/bench_region_tables.py [--scale 1.0] [--steps 20] [--out result.json]
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from bench_large_regions import gpu_identity  # noqa: E402

K0_KERNELS = ("k_signatures", "k_group_insert", "k_group_lookup", "k_group_rank", "k_seq_init", "k_group_region", "k_seq_init_groups")


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of configs[2]'s regions")
    ap.add_argument("--steps", type=int, default=20, help="timed steps per arm")
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--out", default="", help="also write the JSON here")
    args = ap.parse_args()

    import numpy as np
    import torch
    from find_tfbs_b200 import binding, synth
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU fallback")
    torch.cuda.init()
    pats, blk = synth.config3(scale=args.scale)
    ps = binding.PatternSet(pats)
    arms = (("block_tables", 0), ("region_tables", 1))
    ctxs = {}
    for arm, on in arms:
        c = binding.Context(0)
        c.set_option("rows_width", 0)
        c.set_option("region_tables", on)
        c.set_patterns(ps)
        c.upload_block(blk)
        ctxs[arm] = c

    def step(arm):
        c = ctxs[arm]
        t0 = time.perf_counter()
        c.run_resident()
        g = c.collect_grouped()
        return (time.perf_counter() - t0) * 1e3, g, c.stats()

    for _ in range(args.warmup):
        for arm in ctxs:
            step(arm)
    times = {arm: [] for arm in ctxs}
    last = {}
    for _ in range(args.steps):
        for arm in ctxs:
            ms, g, st = step(arm)
            times[arm].append(ms)
            last[arm] = ({k: np.array(v, copy=True) for k, v in g.items() if isinstance(v, np.ndarray)}, st)

    def in_row_order(g):  # the packed words of the rows in row order
        words = (g["n_groups"][g["region"]].astype(np.int64) * g["bits"].astype(np.int64) + 31) // 32
        first = np.repeat(g["offset"].astype(np.int64), words)
        return g["packed"][first + np.arange(int(words.sum())) - np.repeat(np.cumsum(words) - words, words)]

    (g0, st0), (g1, st1) = last["block_tables"], last["region_tables"]
    same = all(np.array_equal(g0[k], g1[k]) for k in ("region", "inner", "pattern_id", "vmin", "vmax", "base", "bits", "n_groups", "hap_group"))
    same = same and np.array_equal(in_row_order(g0), in_row_order(g1))
    counters = ("n_groups", "n_hits", "executed_cells", "evaluated_cells", "n_rows", "n_truncated", "n_dropped")
    same_counters = all(st0[k] == st1[k] for k in counters)

    from torch.profiler import ProfilerActivity, profile
    kernels = {}
    for arm in ctxs:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step(arm)
            torch.cuda.synchronize()
        per = {}
        for ev in prof.key_averages():
            us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
            if us > 0:
                name = ev.key.split("(")[0].split("::")[-1]
                per[name] = per.get(name, 0.0) + us / 1e3
        kernels[arm] = {"k0_kernels_ms": {k: round(v, 4) for k, v in sorted(per.items()) if k.split("<")[0] in K0_KERNELS},
                        "all_kernels_ms": round(sum(per.values()), 3),
                        "top": {k: round(v, 4) for k, v in sorted(per.items(), key=lambda kv: -kv[1])[:16]}}
    for c in ctxs.values():
        c.close()
    out = {
        "gpu": gpu_identity(),
        "workload": "configs[2] (synth.config3, scale %g): %d samples, %d merged regions, %d patterns; block resident, grouped rows, one context per arm" %
                    (args.scale, blk.n_samples, blk.n_regions, ps.n),
        "steps": args.steps,
        "ms_per_step": {arm: {"median": round(statistics.median(t), 3), "mean": round(statistics.mean(t), 3), "min": round(min(t), 3)} for arm, t in times.items()},
        "stages_ms": {arm: {k: round(st[k], 3) for k in ("ms_group", "ms_build", "ms_scan", "ms_count", "ms_total")} for arm, (_, st) in last.items()},
        "launches": {arm: st["total_launches"] for arm, (_, st) in last.items()},
        "kernels_one_step": kernels,
        "rows_identical": bool(same),
        "counters_identical": bool(same_counters),
    }
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
