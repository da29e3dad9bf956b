"""Option "region_tables": the default path groups a region's haplotypes in one CTA's shared memory (k_group_region) instead of the
block-wide tables (k_signatures, k_group_insert, k_group_lookup, k_group_rank), when the block's haplotypes and the records of its
largest region fit there.

Checked here, with region_tables = 0 and = 1 in turn on the same block: the haplotype -> group map, the groups per region, every
array of the grouped rows (the packed counts in row order: where a row's words land is not fixed), the counters of tfbs_stats, and
the attribution, sites and record sites when those options are on are identical, and the rows equal the oracle's.  The shapes:
small cohorts, a configs[2]-like cohort at reduced scale, duplicate records in one region (equal Diff lists under different
carried-record masks), truncations and a sequence-keyed overwrite, a block on each side of the shared-memory limit (where the
block-wide tables must run), reseeded repeats, and signature collisions forced with option test_sig_bits, which both kernels must
detect.
The small cases also run on the emulated kernels (tests/cuda_emu) in the CPU suite."""
import os
import subprocess
import sys

import numpy as np
import pytest

from find_tfbs_b200 import binding, synth
from find_tfbs_b200.binding import PatternSet
import parity_helpers as hp
from test_attribution import rows_packed, truncation_block

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "cuda_emu")
MODES = (binding.ROWS_VARYING, binding.ROWS_ALL_KEYS)
GROUPED = ("region", "inner", "pattern_id", "vmin", "vmax", "base", "bits", "n_groups", "hap_group", "left", "right")
COUNTERS = ("n_regions", "n_groups", "executed_cells", "nominal_cells", "n_hits", "n_keys", "n_rows", "evaluated_cells", "n_scan_items",
            "n_dropped", "n_truncated")
LAUNCHES_SAVED = 3  # k_group_region replaces four launches


def own(x):
    if isinstance(x, dict):
        return {k: own(v) for k, v in x.items() if k != "_c"}
    return np.array(x, copy=True) if isinstance(x, np.ndarray) else x


def run(ps, blk, mode, region_tables, options=None):
    ctx = binding.Context(0)
    try:
        ctx.set_option("rows_mode", mode)
        ctx.set_option("region_tables", region_tables)
        for k, v in (options or {}).items():
            ctx.set_option(k, v)
        ctx.set_patterns(ps)
        ctx.submit_block(blk)
        out = {"grouped": own(ctx.collect_grouped(expand=True)), "stats": ctx.stats()}
        if (options or {}).get("attribution"):
            out["attribution"] = own(ctx.attribution())
        if (options or {}).get("sites"):
            out["sites"] = own(ctx.sites())
        if (options or {}).get("record_sites"):
            out["record_sites"] = own(ctx.record_sites())
        return out
    finally:
        ctx.close()


def assert_same(a, b, what):
    if isinstance(a, dict):
        assert a.keys() == b.keys(), what
        for k in a:
            assert_same(a[k], b[k], what + "." + k)
    elif isinstance(a, np.ndarray):
        assert a.dtype == b.dtype and np.array_equal(a, b), what
    else:
        assert a == b, what


def check(ps, blk, options=None, modes=MODES, fits=True):
    """Both settings of the option on one block in each row mode: identical outputs, rows equal to the oracle's; `fits` says whether
    region_tables = 1 took the shared-memory kernel (three launches fewer) or the block-wide tables (the same launches)."""
    for mode in modes:
        o = hp.run_oracle(ps, blk, mode)
        old = run(ps, blk, mode, 0, options)
        new = run(ps, blk, mode, 1, options)
        for k in GROUPED:
            assert_same(old["grouped"][k], new["grouped"][k], k)
        assert_same(rows_packed(old["grouped"]), rows_packed(new["grouped"]), "packed")
        for k in ("attribution", "sites", "record_sites"):
            if k in old:
                assert_same(old[k], new[k], k)
        for k in COUNTERS:
            assert old["stats"][k] == new["stats"][k], k
        hp.assert_rows_equal(new["grouped"], o)
        hp.check_stats(new["stats"], o)
        saved = old["stats"]["total_launches"] - new["stats"]["total_launches"]
        assert saved == (LAUNCHES_SAVED if fits else 0), saved
    return new


def small_cohort(seed, n_samples=12, n_regions=40):
    pats = synth.make_pwms(6, seed=seed, lmin=4, lmax=30)
    lmax = max(p["weights"].shape[0] for p in pats)
    return PatternSet(pats), synth.make_cohort(n_samples, n_regions, seed=seed, lmax_pattern=lmax, region_len=(50, 600), variant_rate=1 / 20.0,
                                               same_pos_frac=0.05)


def duplicate_records_block():
    """Region 0 holds the same Diff (pos 10, G -> A) twice and (pos 14, G -> GAC) twice, carried by different haplotypes: haplotypes
    with equal Diff lists but different carried-record masks, which one group must hold; region 1 has no duplicates."""
    g = "ACGTACGTACGTACGTACGTACGT"
    blk = hp.hand_block(6, [(0, 23, g), (2, 15, g[2:16])],
                        [(0, 10, "G", "A"), (0, 10, "G", "A"), (0, 14, "G", "GAC"), (0, 14, "G", "GAC"), (0, 3, "T", "C"),
                         (1, 5, "C", "T"), (1, 9, "C", "G")],
                        [[0, 3, 7], [1, 4, 8], [0, 5, 9], [1, 2, 10], [0, 1, 2, 3, 11], [0, 1], [2, 3, 4]])
    w = np.array([[1000, 0, 0, 0], [0, 1000, 0, 0]], dtype=np.int32)
    ps = PatternSet([{"weights": w, "min_score": 1500, "pattern_id": 7}, {"weights": w[::-1, ::-1].copy(), "min_score": 1500, "pattern_id": 7, "direction": 1}])
    return ps, blk


# ---- small cases (GPU and emulated kernels) ---------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2])
def test_small_cohort(seed):
    ps, blk = small_cohort(seed)
    check(ps, blk)


@pytest.mark.gpu
def test_small_duplicate_records():
    ps, blk = duplicate_records_block()
    new = check(ps, blk)
    hg = new["grouped"]["hap_group"]
    # haplotype 0 carries records 0, 2, 4 and haplotype 1 records 1, 3, 4: the same Diff list under different masks
    assert hg[0, 0] == hg[0, 1] and hg[0, 0] != 0


@pytest.mark.gpu
def test_small_truncation_and_overwrite():
    ps, blk = truncation_block()
    check(ps, blk)


@pytest.mark.gpu
def test_small_attribution_sites_record_sites():
    ps, blk = small_cohort(3)
    check(ps, blk, options={"attribution": 1, "sites": 1, "record_sites": 1})
    ps, blk = truncation_block()
    check(ps, blk, options={"attribution": 1, "sites": 1, "record_sites": 1})


@pytest.mark.gpu
def test_small_reseeded_repeat():
    """Option test_reseed treats the first attempt of every block as a hash collision: the repeat with another seed runs the
    shared-memory kernel again and gives the same result."""
    ps, blk = small_cohort(4)
    check(ps, blk, options={"test_reseed": 1}, modes=(binding.ROWS_VARYING,))


@pytest.mark.gpu
def test_small_forced_signature_collision():
    """Option test_sig_bits = 1 gives every carrier haplotype of the first attempt the same signature: one table slot holds different
    diff lists.  With the exact check on (verify_groups, the default) both kernels count the collision and the block is repeated with
    full signatures: groups and rows equal the oracle's.  With the check off nothing repeats and the merged groups come out, which
    shows that the first attempt did meet collisions."""
    ps, blk = small_cohort(5)
    o = hp.run_oracle(ps, blk, binding.ROWS_VARYING)
    for region_tables in (0, 1):
        good = run(ps, blk, binding.ROWS_VARYING, region_tables, {"test_sig_bits": 1})
        hp.assert_rows_equal(good["grouped"], o)
        hp.check_stats(good["stats"], o)
        merged = run(ps, blk, binding.ROWS_VARYING, region_tables, {"test_sig_bits": 1, "verify_groups": 0})
        assert merged["stats"]["n_groups"] < o["n_groups"], region_tables
    assert_same(good["grouped"]["hap_group"], run(ps, blk, binding.ROWS_VARYING, 0, {"test_sig_bits": 1})["grouped"]["hap_group"], "hap_group")


# ---- larger shapes (GPU only) -------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_configs2_like_cohort():
    """configs[2]'s shape at reduced scale: 2,504 samples, two BED sets, 401 PWMs cut to 40, haplotypes shared in LD blocks."""
    pats = synth.make_pwms(40, seed=21, lmin=6, lmax=21)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(2504, 24, seed=21, lmax_pattern=lmax, region_len=(200, 1500), two_beds=True, ld_blocks=64)
    check(PatternSet(pats), blk, options={"attribution": 1, "sites": 1})


@pytest.mark.gpu
@pytest.mark.parametrize("n_samples,fits", [(3200, True), (3300, False)])
def test_both_sides_of_the_shared_memory_limit(n_samples, fits):
    """6,400 haplotypes fit an 8,192-slot table next to their counters and masks; 6,600 need 16,384 slots, which do not fit: the
    block-wide tables run."""
    pats = synth.make_pwms(6, seed=5, lmin=6, lmax=16)
    blk = synth.make_cohort(n_samples, 6, seed=5, lmax_pattern=16, region_len=(200, 600), variant_rate=1 / 40.0, ld_blocks=200)
    check(PatternSet(pats), blk, modes=(binding.ROWS_VARYING,), fits=fits)


# ---- the small cases on the emulated kernels (CPU) ----------------------------------------------------------------------------------

def test_small_cases_on_emulated_kernels():
    subprocess.check_call(["make", "-C", EMU, "-j2", "libtfbs_emu.so"], stdout=subprocess.DEVNULL)
    env = dict(os.environ, TFBS_B200_LIB=os.path.join(EMU, "libtfbs_emu.so"))
    cmd = [sys.executable, "-m", "pytest", "tests/test_region_tables.py", "-q", "-x", "-m", "gpu", "-k", "small", "-p", "no:cacheprovider"]
    r = subprocess.run(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-4000:]
    assert "7 passed" in r.stdout, r.stdout[-2000:]
