#!/usr/bin/env python
"""What option "attribution" costs on the BASELINE.json configs[2] block (synth.config3: 2,504 samples, two BED sets, 401 PWMs on
both strands), the shape bench.py measures.  Two contexts in one process, option off and on, each with the block resident in HBM
(tfbs_upload_block once, tfbs_run_resident per step); the steps alternate between them.  A step ends with the grouped rows on the host
(tfbs_collect_grouped, which in the "on" arm also copies the attribution to the host) and tfbs_get_attribution; it is timed with the
host clock.

Reported per arm: ms per step (median and mean), ms_total (device time of the run, tfbs_stats) and device -> host bytes; for the on
arm: the extra bytes tfbs_get_attribution copies, terms / configurations / group-list entries per step, the extra kernel launches, and
the device time of the k_att_* kernels in one step (torch.profiler; the four scans and the gate that the attribution also launches
share their kernels with the rest of the pipeline and are not in that sum -- the ms_total difference covers them).  The off arm's rows
are compared with the on arm's.  The card's name and power limit are read in the same run.

  python scripts/bench_attribution.py [--scale 1.0] [--steps 10] [--out result.json]
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


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of configs[2]'s regions")
    ap.add_argument("--steps", type=int, default=10, help="timed steps per arm")
    ap.add_argument("--warmup", type=int, default=3)
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
    ctxs = {}
    for arm, on in (("off", 0), ("on", 1)):
        c = binding.Context(0)
        c.set_option("rows_width", 0)
        c.set_option("attribution", on)
        c.set_patterns(ps)
        c.upload_block(blk)
        ctxs[arm] = c

    import ctypes as C

    def step(arm):  # the attribution is fetched through the C call alone: the binding's NumPy copies are not part of the step
        c = ctxs[arm]
        t0 = time.perf_counter()
        c.run_resident()
        g = c.collect_grouped()
        if arm == "on":
            raw = binding.TfbsAttribution()
            if c._lib.tfbs_get_attribution(c._h, C.byref(raw)) != binding.TFBS_OK:
                raise SystemExit("tfbs_get_attribution failed")
        ms = (time.perf_counter() - t0) * 1e3
        return ms, g, None, c.stats()

    for _ in range(args.warmup):
        for arm in ctxs:
            step(arm)
    times = {arm: [] for arm in ctxs}
    last = {}
    for _ in range(args.steps):
        for arm in ctxs:
            ms, g, a, st = step(arm)
            times[arm].append(ms)
            last[arm] = (g, a, st)
    g_off, _, st_off = last["off"]
    g_on, _, st_on = last["on"]
    a = ctxs["on"].attribution()  # the last step's attribution as arrays (already on the host: no second copy)

    def in_row_order(g):  # the packed words of the rows in row order (the payload order in `packed` is not fixed)
        words = (g["n_groups"][g["region"]].astype(np.int64) * g["bits"].astype(np.int64) + 31) // 32
        first = np.repeat(g["offset"].astype(np.int64), words)
        return g["packed"][first + np.arange(int(words.sum())) - np.repeat(np.cumsum(words) - words, words)]

    same = all(np.array_equal(g_off[k], g_on[k]) for k in ("region", "inner", "pattern_id", "vmin", "vmax", "base", "bits", "n_groups", "hap_group"))
    same = same and np.array_equal(in_row_order(g_off), in_row_order(g_on))

    # device time of the k_att_* kernels of one step of the on arm
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step("on")
        torch.cuda.synchronize()
    att_us, att_n = 0.0, 0
    for ev in prof.key_averages():
        if "k_att_" in ev.key:
            att_us += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
            att_n += ev.count

    for c in ctxs.values():
        c.close()
    out = {
        "gpu": gpu_identity(),
        "workload": "configs[2] (synth.config3, scale %g): %d samples, %d merged regions, %d patterns; block resident, grouped rows" %
                    (args.scale, blk.n_samples, blk.n_regions, ps.n),
        "steps": args.steps,
        "ms_per_step": {arm: {"median": round(statistics.median(t), 3), "mean": round(statistics.mean(t), 3), "min": round(min(t), 3)} for arm, t in times.items()},
        "ms_total_device": {"off": round(st_off["ms_total"], 3), "on": round(st_on["ms_total"], 3)},
        "ms_count_device": {"off": round(st_off["ms_count"], 3), "on": round(st_on["ms_count"], 3)},
        "k_att_kernels_device_ms": round(att_us / 1e3, 4),
        "k_att_kernel_launches": att_n,
        "extra_launches": st_on["total_launches"] - st_off["total_launches"],
        "d2h_bytes": {"off": st_off["d2h_bytes"], "on": st_on["d2h_bytes"], "on_attribution_extra": st_on["d2h_bytes"] - st_off["d2h_bytes"]},
        "rows": int(a["n_rows"]),
        "terms": int(len(a["term_cfg"])),
        "configurations": int(a["n_cfgs"]),
        "group_list_entries": int(len(a["group_cfg"])),
        "groups": int(a["n_groups_total"]),
        "rows_identical_off_on": bool(same),
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
