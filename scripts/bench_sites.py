#!/usr/bin/env python
"""What option "sites" costs on the BASELINE.json configs[2] block (synth.config3: 2,504 samples, two BED sets, 401 PWMs on both
strands), the shape bench.py measures.  Two contexts in one process, both with option "attribution" = 1, one also with "sites" = 1,
each with the block resident in HBM (tfbs_upload_block once, tfbs_run_resident per step); the steps alternate between them.  A step
ends with the grouped rows on the host (tfbs_collect_grouped, which also copies the attribution, and in the sites arm the sites, to
the host) and the C calls tfbs_get_attribution / tfbs_get_sites; it is timed with the host clock.

Reported per arm: ms per step (median, mean, min), ms_total and ms_scan_kernel (device time of the run and of the scan launches,
tfbs_stats) and device -> host bytes; for the sites arm: the extra launches and bytes, gained / lost sites per step, and the device
time of the k_site_* kernels in one step (torch.profiler; the scoring in the scan's rare path is inside ms_scan_kernel, the two
scans and gates share their kernels with the rest of the pipeline and are covered by the ms_total difference).  The rows and the
attribution of the two arms are compared.  The card's name and power limit are read in the same run.

  python scripts/bench_sites.py [--scale 1.0] [--steps 10] [--out result.json]
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
    for arm, on in (("attribution", 0), ("sites", 1)):
        c = binding.Context(0)
        c.set_option("rows_width", 0)
        c.set_option("attribution", 1)
        c.set_option("sites", on)
        c.set_patterns(ps)
        c.upload_block(blk)
        ctxs[arm] = c

    def step(arm):  # attribution and sites are fetched through the C calls alone: the binding's NumPy copies are not part of the step
        c = ctxs[arm]
        t0 = time.perf_counter()
        c.run_resident()
        g = c.collect_grouped()
        if c._lib.tfbs_get_attribution(c._h, C.byref(binding.TfbsAttribution())) != binding.TFBS_OK:
            raise SystemExit("tfbs_get_attribution failed")
        if arm == "sites" and c._lib.tfbs_get_sites(c._h, C.byref(binding.TfbsSites())) != binding.TFBS_OK:
            raise SystemExit("tfbs_get_sites failed")
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
    g0, st0 = last["attribution"]
    g1, st1 = last["sites"]
    a0, a1 = ctxs["attribution"].attribution(), ctxs["sites"].attribution()
    s = ctxs["sites"].sites()

    def in_row_order(g):  # the packed words of the rows in row order (the payload order in `packed` is not fixed)
        words = (g["n_groups"][g["region"]].astype(np.int64) * g["bits"].astype(np.int64) + 31) // 32
        first = np.repeat(g["offset"].astype(np.int64), words)
        return g["packed"][first + np.arange(int(words.sum())) - np.repeat(np.cumsum(words) - words, words)]

    same_rows = all(np.array_equal(g0[k], g1[k]) for k in ("region", "inner", "pattern_id", "vmin", "vmax", "base", "bits", "n_groups", "hap_group"))
    same_rows = same_rows and np.array_equal(in_row_order(g0), in_row_order(g1))
    same_att = all(np.array_equal(a0[k], a1[k]) for k in a0 if isinstance(a0[k], np.ndarray))

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step("sites")
        torch.cuda.synchronize()
    site_us, site_n = 0.0, 0
    for ev in prof.key_averages():
        if "k_site_" in ev.key:
            site_us += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
            site_n += ev.count

    for c in ctxs.values():
        c.close()
    out = {
        "gpu": gpu_identity(),
        "workload": "configs[2] (synth.config3, scale %g): %d samples, %d merged regions, %d patterns; block resident, grouped rows, "
                    "attribution on in both arms" % (args.scale, blk.n_samples, blk.n_regions, ps.n),
        "steps": args.steps,
        "ms_per_step": {arm: {"median": round(statistics.median(t), 3), "mean": round(statistics.mean(t), 3), "min": round(min(t), 3)} for arm, t in times.items()},
        "ms_total_device": {"attribution": round(st0["ms_total"], 3), "sites": round(st1["ms_total"], 3)},
        "ms_scan_kernel_device": {"attribution": round(st0["ms_scan_kernel"], 3), "sites": round(st1["ms_scan_kernel"], 3)},
        "k_site_kernels_device_ms": round(site_us / 1e3, 4),
        "k_site_kernel_launches": site_n,
        "extra_launches": st1["total_launches"] - st0["total_launches"],
        "d2h_bytes": {"attribution": st0["d2h_bytes"], "sites": st1["d2h_bytes"], "sites_extra": st1["d2h_bytes"] - st0["d2h_bytes"]},
        "configurations": int(s["n_cfgs"]),
        "sites_gained": int((s["change"] > 0).sum()),
        "sites_lost": int((s["change"] < 0).sum()),
        "rows_identical": bool(same_rows),
        "attribution_identical": bool(same_att),
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
