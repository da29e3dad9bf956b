#!/usr/bin/env python
"""What option "record_sites" costs on the BASELINE.json configs[2] block (synth.config3: 2,504 samples, two BED sets, 401 PWMs on
both strands), the shape bench.py measures.  Two contexts in one process, one with "record_sites" = 0 and one with 1 (attribution
and sites off in both), each with the block resident in HBM (tfbs_upload_block once, tfbs_run_resident per step); the steps
alternate between them.  A step ends with the grouped rows on the host (tfbs_collect_grouped, which in the record arm also copies
the record sites) and, in the record arm, the C call tfbs_get_record_sites; it is timed with the host clock.

Reported per arm: ms per step (median, mean, min), ms_total and ms_scan_kernel (device time of the run and of the scan launches,
tfbs_stats) and device -> host bytes; for the record arm: the extra launches and bytes, records, flagged records and gained / lost
sites per step, and the device time of the k_site_* kernels in one step (torch.profiler, a run of its own; the scoring of the
records' windows is inside ms_scan_kernel).  The rows of the two arms are compared.  The card's name and power limit are read in the
same run.

  python scripts/bench_record_sites.py [--scale 1.0] [--steps 10] [--out result.json]
"""
import argparse
import ctypes as C
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
    for arm, on in (("off", 0), ("record_sites", 1)):
        c = binding.Context(0)
        c.set_option("rows_width", 0)
        c.set_option("record_sites", on)
        c.set_patterns(ps)
        c.upload_block(blk)
        ctxs[arm] = c

    def step(arm):  # the record sites are fetched through the C call alone: the binding's NumPy copies are not part of the step
        c = ctxs[arm]
        t0 = time.perf_counter()
        c.run_resident()
        g = c.collect_grouped()
        if arm == "record_sites" and c._lib.tfbs_get_record_sites(c._h, C.byref(binding.TfbsRecordSites())) != binding.TFBS_OK:
            raise SystemExit("tfbs_get_record_sites failed")
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
            last[arm] = (g, st)
    g0, st0 = last["off"]
    g1, st1 = last["record_sites"]
    rs = ctxs["record_sites"].record_sites()

    def in_row_order(g):  # the packed words of the rows in row order (the payload order in `packed` is not fixed)
        words = (g["n_groups"][g["region"]].astype(np.int64) * g["bits"].astype(np.int64) + 31) // 32
        first = np.repeat(g["offset"].astype(np.int64), words)
        return g["packed"][first + np.arange(int(words.sum())) - np.repeat(np.cumsum(words) - words, words)]

    same_rows = all(np.array_equal(g0[k], g1[k]) for k in ("region", "inner", "pattern_id", "vmin", "vmax", "base", "bits", "n_groups", "hap_group"))
    same_rows = same_rows and np.array_equal(in_row_order(g0), in_row_order(g1))

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step("record_sites")
        torch.cuda.synchronize()
    site_us, site_n = 0.0, 0
    for ev in prof.key_averages():
        if "k_site_" in ev.key:
            site_us += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
            site_n += ev.count

    for c in ctxs.values():
        c.close()
    fl = rs["rec_flags"]
    out = {
        "gpu": gpu_identity(),
        "workload": "configs[2] (synth.config3, scale %g): %d samples, %d merged regions, %d patterns; block resident, grouped rows, "
                    "attribution and sites off in both arms" % (args.scale, blk.n_samples, blk.n_regions, ps.n),
        "steps": args.steps,
        "ms_per_step": {arm: {"median": round(statistics.median(t), 3), "mean": round(statistics.mean(t), 3), "min": round(min(t), 3)} for arm, t in times.items()},
        "ms_total_device": {"off": round(st0["ms_total"], 3), "record_sites": round(st1["ms_total"], 3)},
        "ms_scan_kernel_device": {"off": round(st0["ms_scan_kernel"], 3), "record_sites": round(st1["ms_scan_kernel"], 3)},
        "k_site_kernels_device_ms": round(site_us / 1e3, 4),
        "k_site_kernel_launches": site_n,
        "extra_launches": st1["total_launches"] - st0["total_launches"],
        "scan_launches": {"off": st0["scan_launches"], "record_sites": st1["scan_launches"]},
        "d2h_bytes": {"off": st0["d2h_bytes"], "record_sites": st1["d2h_bytes"], "extra": st1["d2h_bytes"] - st0["d2h_bytes"]},
        "records": int(rs["n_records"]),
        "records_flagged": {"outside": int((fl & binding.REC_OUTSIDE != 0).sum()), "ref_mismatch": int((fl & binding.REC_REF_MISMATCH != 0).sum()),
                            "missing_case": int((fl & binding.REC_MISSING_CASE != 0).sum())},
        "sites_gained": int((rs["change"] > 0).sum()),
        "sites_lost": int((rs["change"] < 0).sum()),
        "rows_identical": bool(same_rows),
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
