"""Regions with more distinct haplotypes than the fan-out's shared-memory count vector holds (53,120 groups): dense biobank
cohorts, where nearly every haplotype of a region is distinct.  The fan-out then keeps one count vector per CTA in device memory
(k_fanout<true>); the rows must not change.

On the GPU: a 40,000-sample dense cohort whose largest region has more than 65,536 groups (4-byte haplotype -> group map, rows
wider than the staging buffer) against the oracle on the whole cohort, through the dense and the grouped results, one context
started cold, and the C++ driver; the same cohort in two sample blocks; a region just below the shared-memory capacity in a block
that could have more groups; and the device-memory vector forced onto small shapes (option fan_vector = 1) through the parity
machinery.

On the CPU: the forced cases run again on the emulated kernels (tests/cuda_emu), and a debug build of the emulated library counts
the keys of the dense pass on the many-keys shape.  The 30,000- and 40,000-sample cases are too large for the emulator and are left
out of that run with -k."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from find_tfbs_b200 import binding, sharding, synth
from find_tfbs_b200.binding import PatternSet
from oracle import pyoracle as ora
import file_writers as fw
import parity_helpers as hp
from test_gpu_parity import acgt_patterns, fixture_block

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "cuda_emu")
SMEM_GROUPS = 53120  # groups the shared-memory count vector holds (227 KB a block less the static shared memory, the pairs and the staging buffer)
FAN_STAGE = 1024     # packed words a CTA stages in shared memory; wider rows are written out directly
MODES = (binding.ROWS_VARYING, binding.ROWS_ALL_KEYS)


# ---- the large cohort: 40,000 samples, a record every ~4 bp, two regions of 500-700 bp --------------------------------------

@pytest.fixture(scope="module")
def large():
    """Seed 5: region 0 has 79,998 groups and no sequence-keyed overwrite, region 1 has 76,125 groups and one overwrite."""
    pats = synth.make_pwms(4, seed=5, lmin=6, lmax=10, pvalue=1e-3)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(40000, 2, seed=5, lmax_pattern=lmax, region_len=(500, 700), variant_rate=1 / 4.0, gap=(100, 300))
    return pats, PatternSet(pats), blk


@pytest.fixture(scope="module")
def large_oracle(large):
    _, ps, blk = large
    return {mode: hp.run_oracle(ps, blk, mode, False, os.cpu_count() or 4, 1) for mode in MODES}


def region_rows(o, blk, r):
    """Rows of region r of a whole-block result, renumbered as the result of the block blk.slice(r, r + 1)."""
    sel = np.nonzero(o["region"] == r)[0]
    out = {k: o[k][sel] for k in ("pattern_id", "vmin", "vmax", "left", "right")}
    out["region"] = o["region"][sel] - r
    out["inner"] = o["inner"][sel] - int(blk.inner_off[r])
    return out


@pytest.mark.gpu
def test_region_beyond_shared_memory(large, large_oracle):
    """Regions of 79,998 and 76,125 groups: dense rows (tfbs_collect) and grouped rows expanded on the host (tfbs_collect_grouped +
    tfbs_expand_rows) equal the whole-cohort oracle in both row modes, counters included; the map comes back with 4-byte entries
    and every varying row is wider than the staging buffer."""
    _, ps, blk = large
    for mode in MODES:
        o = large_oracle[mode]
        assert len(o["region"]) > 0
        d = hp.run_gpu(ps, blk, mode)
        hp.assert_rows_equal(d, o)
        hp.check_stats(d["stats"], o)
        ctx = binding.Context(0)
        try:
            ctx.set_option("rows_mode", mode)
            ctx.set_patterns(ps)
            ctx.submit_block(blk)
            g = ctx.collect_grouped(expand=True)
            st = ctx.stats()
            hp.assert_rows_equal(g, o)
            hp.check_stats(st, o)
            assert int(g["n_groups"].max()) > 65536 > SMEM_GROUPS
            assert g["_c"].hap_group_bytes == 4 and g["hap_group"].dtype == np.uint32
            assert int(g["hap_group"].max()) >= 65536  # group numbers that do not fit the 2-byte map
            words = (g["n_groups"][g["region"]].astype(np.int64) * g["bits"] + 31) // 32
            assert (words > FAN_STAGE).any()
        finally:
            ctx.close()


@pytest.mark.gpu
def test_one_block_vs_sample_blocks(large, large_oracle):
    """Each region as one block of 40,000 samples (count vector in device memory) and as two sample blocks of 20,000 (shared
    memory) merged by tfbs_merge_sample_blocks: the same rows where no sequence-keyed overwrite happened.  Where one happened (the
    winner is chosen per block), the single block still equals the whole-cohort oracle."""
    _, ps, blk = large
    o = large_oracle[binding.ROWS_VARYING]
    checked = {"merged": 0, "overwrite": 0}
    for r in range(blk.n_regions):
        one = blk.slice(r, r + 1)
        single = hp.run_gpu(ps, one)
        hp.assert_rows_equal(single, region_rows(o, blk, r))
        ctx = binding.Context(0)
        try:
            ctx.set_option("rows_mode", binding.ROWS_ALL_KEYS)
            ctx.set_patterns(ps)
            parts, dropped = [], single["stats"]["n_dropped"]
            for a, b in ((0, 20000), (20000, 40000)):
                ctx.submit_block(sharding.sample_block(one, a, b))
                parts.append(binding.own_grouped(ctx.collect_grouped()))
                assert int(parts[-1]["n_groups"].max()) <= SMEM_GROUPS
                dropped += ctx.stats()["n_dropped"]
        finally:
            ctx.close()
        merged = binding.merge_sample_blocks(parts)
        if dropped == 0:
            hp.assert_rows_equal(merged, single)
            checked["merged"] += 1
        else:
            checked["overwrite"] += 1
    assert checked == {"merged": 1, "overwrite": 1}


@pytest.mark.gpu
def test_region_at_the_shared_memory_capacity():
    """30,000 samples (up to 60,001 groups per region: more than shared memory holds) and a largest region of 51,951 groups: the
    capacity with its 25 % slack would not fit shared memory, so it is clamped to the shared-memory capacity and the fan-out runs in
    shared memory with the largest count vector the device allows next to the kernel's static shared memory.  The first block of a
    cold context grows into that capacity, the second starts from it (the context's hint)."""
    pats = synth.make_pwms(4, seed=6, lmin=6, lmax=10, pvalue=1e-3)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(30000, 2, seed=6, lmax_pattern=lmax, region_len=(350, 450), variant_rate=1 / 4.0, gap=(100, 300))
    ps = PatternSet(pats)
    o = hp.run_oracle(ps, blk, binding.ROWS_ALL_KEYS, False, os.cpu_count() or 4, 1)
    ctx = binding.Context(0)
    try:
        ctx.set_option("rows_mode", binding.ROWS_ALL_KEYS)
        ctx.set_patterns(ps)
        ctx.submit_block(blk)
        hp.assert_rows_equal(ctx.collect(), o)
        hp.check_stats(ctx.stats(), o)
        ctx.submit_block(blk)
        g = ctx.collect_grouped(expand=True)
        hp.assert_rows_equal(g, o)
        ng = int(g["n_groups"].max())
        assert 2 * blk.n_samples + 1 > SMEM_GROUPS >= ng and ng + ng // 4 + 16 > SMEM_GROUPS
    finally:
        ctx.close()


@pytest.mark.gpu
def test_cold_context_grows_into_device_memory(large, large_oracle):
    """The first block of a fresh context is the large cohort: the fan-out starts from a guess of 2,048 groups, asks for more and the
    block is repeated with the count vectors in device memory.  A small block submitted next on the same context is still right."""
    _, ps, blk = large
    small_pats = synth.make_pwms(5, seed=41)
    small = synth.make_cohort(16, 12, seed=41, lmax_pattern=max(p["weights"].shape[0] for p in small_pats), region_len=(100, 600))
    ctx = binding.Context(0)
    try:
        ctx.set_patterns(ps)
        ctx.submit_block(blk)
        d = ctx.collect()
        hp.assert_rows_equal(d, large_oracle[binding.ROWS_VARYING])
        hp.check_stats(ctx.stats(), large_oracle[binding.ROWS_VARYING])
        sps = PatternSet(small_pats)
        ctx.set_patterns(sps)
        ctx.submit_block(small)
        hp.assert_rows_equal(ctx.collect(), hp.run_oracle(sps, small))
    finally:
        ctx.close()


@pytest.mark.gpu
def test_driver_on_large_regions(large, tmp_path):
    """find-tfbs-b200 on the large cohort written as files (BCF of 40,000 samples): the VCF equals the oracle's run() on the same files,
    with the default options and with one region per block on two contexts."""
    import test_driver as td
    pats, _, blk = large
    a = fw.cohort_to_files(blk, pats, str(tmp_path))
    expected = ora.run(a["chromosome"], a["bcf"], a["beds"], a["reference"], None, a["pwm_file"], a["threshold_dir"], 1e-4, a["names"],
                       threads=os.cpu_count() or 4)
    assert len(expected.splitlines()) > 1
    for extra in ([], ["--chunk", "1", "--devices", "0,0"]):
        out = str(tmp_path / "out.vcf.gz")
        a["extra"] = extra
        p = td.run_driver(a, out)
        assert p.returncode == 0, p.stderr
        assert ora.gunzip_file(out) == expected


# ---- the device-memory count vector forced onto small shapes (option fan_vector = 1) ---------------------------------------------

def forced_equal(ps, blk, mode, options=None, o=None):
    """Default path, forced device-memory vector and oracle: the same rows, the same counters, the same count width."""
    o = hp.run_oracle(ps, blk, mode) if o is None else o
    base = hp.run_gpu(ps, blk, mode, options=options)
    vec = hp.run_gpu(ps, blk, mode, options=dict(options or {}, fan_vector=1))
    hp.assert_rows_equal(base, o)
    hp.assert_rows_equal(vec, o)
    assert vec["count_bytes"] == base["count_bytes"]
    assert vec["left"].tobytes() == base["left"].tobytes() and vec["right"].tobytes() == base["right"].tobytes()
    hp.check_stats(vec["stats"], o)
    return vec, o


@pytest.mark.gpu
def test_forced_device_vector_fixture():
    """The reference's integration fixture (one SNV carried by one haplotype) in both row modes."""
    vec, _ = forced_equal(acgt_patterns(), fixture_block([0]), binding.ROWS_VARYING)
    assert (vec["left"][0] + vec["right"][0]).tolist() == [2, 4, 4, 4]
    forced_equal(acgt_patterns(), fixture_block([0]), binding.ROWS_ALL_KEYS)


@pytest.mark.gpu
def test_forced_device_vector_threshold_ties():
    """Thresholds at and next to attainable scores (strict >, pattern.rs:151)."""
    rng = np.random.default_rng(3)
    w = rng.integers(-3, 4, size=(8, 4)).astype(np.int32) * 100
    blk = synth.make_cohort(6, 20, seed=9, lmax_pattern=8, region_len=(200, 400))
    best = int(w.max(axis=1).sum())
    for ms in (best - 401, best - 400, best - 300):
        forced_equal(PatternSet([{"weights": w, "min_score": ms, "pattern_id": 1}]), blk, binding.ROWS_ALL_KEYS)


def many_keys_case():
    """40 patterns x several inner regions per region on a dense cohort: rounds of many keys with differences, so that the pairs of a
    round overflow the FAN_PAIRS kept in shared memory and later keys take the dense pass."""
    pats = synth.make_pwms(40, seed=17, lmin=6, lmax=12, pvalue=5e-3)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(120, 3, seed=17, lmax_pattern=lmax, region_len=(300, 500), variant_rate=1 / 4.0, gap=(100, 300), two_beds=True)
    return PatternSet(pats), blk


@pytest.mark.gpu
def test_forced_device_vector_many_keys():
    ps, blk = many_keys_case()
    for mode in MODES:
        _, o = forced_equal(ps, blk, mode)
        assert len(o["region"]) > 0


def test_many_keys_case_runs_both_passes(tmp_path):
    """The many-keys shape reaches the sparse and the dense pass of the device-memory fan-out: the emulated library built with
    -DTFBS_FAN_STATS counts the keys with a count vector and, among them, the keys of the dense pass (TFBS_DEBUG prints both)."""
    lib = str(tmp_path / "libtfbs_emu_stats.so")
    csrc = os.path.join(ROOT, "find_tfbs_b200", "csrc")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-pthread", "-w", "-DTFBS_FAN_STATS", "-shared", "-I", os.path.join(EMU, "include"),
                           "-x", "c++", os.path.join(csrc, "tfbs.cu"), os.path.join(csrc, "tables.cpp"), "-o", lib])
    env = dict(os.environ, TFBS_B200_LIB=lib, TFBS_DEBUG="1", PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "tests")]))
    code = ("import parity_helpers as hp, test_large_regions as t\n"
            "ps, blk = t.many_keys_case()\n"
            "hp.run_gpu(ps, blk, 0, options={'fan_vector': 1})\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    m = re.search(r"fan-out: (\d+) keys with a count vector.*, (\d+) keys in the dense pass", r.stderr)
    assert m, r.stderr[-3000:]
    heavy, dense = int(m.group(1)), int(m.group(2))
    assert 0 < dense < heavy, (heavy, dense)


@pytest.mark.gpu
def test_forced_device_vector_tiny_caps_and_narrow_rows():
    """Option tiny_caps (every capacity, the count vector's included, grows through repeated runs) and option rows_width = 0."""
    pats = synth.make_pwms(6, seed=2)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(12, 10, seed=2, lmax_pattern=lmax, region_len=(200, 600), two_beds=True, n_runs=2, same_pos_frac=0.1,
                            frac_ins=0.15, frac_del=0.15)
    ps = PatternSet(pats)
    for mode in MODES:
        o = hp.run_oracle(ps, blk, mode)
        forced_equal(ps, blk, mode, {"tiny_caps": 1}, o)
        forced_equal(ps, blk, mode, {"rows_width": 0}, o)


@pytest.mark.gpu
def test_forced_device_vector_in_flight_twin_and_arena():
    """Two blocks in flight on one lane and, with option dual_stream, on two lanes (each with its own count vectors), grouped rows
    expanded on the host, and a result arena whose halves are written by the two lanes."""
    pats = synth.make_pwms(6, seed=3)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(12, 10, seed=3, lmax_pattern=lmax, region_len=(200, 600), two_beds=True, frac_ins=0.15, frac_del=0.15)
    ps = PatternSet(pats)
    half = blk.n_regions // 2
    b1, b2 = blk.slice(0, half), blk.slice(half, blk.n_regions)
    for mode in MODES:
        o1, o2 = hp.run_oracle(ps, b1, mode), hp.run_oracle(ps, b2, mode)
        for dual in (0, 1):
            ctx = binding.Context(0)
            try:
                ctx.set_option("rows_mode", mode)
                with pytest.raises(binding.TfbsError):
                    ctx.set_option("fan_vector", 2)
                ctx.set_option("fan_vector", 1)
                ctx.set_patterns(ps)
                ctx.set_option("dual_stream", dual)
                ctx.submit_block(b1)
                ctx.submit_block(b2)
                g1 = binding.own_grouped(ctx.collect_grouped(expand=True))
                g2 = ctx.collect_grouped(expand=True)
                hp.assert_rows_equal(g1, o1)
                hp.assert_rows_equal(g2, o2)
                if dual:
                    raw = np.zeros((4 << 20) + 64, dtype=np.uint8)
                    arena = raw[(-raw.ctypes.data) % 64:][:4 << 20]  # 64-byte aligned
                    ctx.set_result_arena(arena)
                    for b in (b1, b2):
                        ctx.submit_block(b)
                        ctx.collect_grouped()
                    hp.assert_rows_equal(binding.read_arena(arena, 0, expand=True), o1)
                    hp.assert_rows_equal(binding.read_arena(arena, 1, expand=True), o2)
                    ctx.set_result_arena(None)
            finally:
                ctx.close()


# ---- the forced cases on the emulated kernels (CPU) -------------------------------------------------------------------------------

def run_marked_gpu_tests(env, path, select, workers=4):
    cmd = [sys.executable, "-m", "pytest", path, "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider"]
    try:
        import xdist  # noqa: F401  (the emulation is single-threaded per process: spread the cases over a few processes)
        cmd += ["-n", str(workers)]
    except ImportError:
        pass
    if select:
        cmd += ["-k", select]
    r = subprocess.run(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-4000:]
    assert " passed" in r.stdout and "failed" not in r.stdout
    return r.stdout


def test_forced_device_vector_on_emulated_kernels():
    """The forced device-memory cases above on tests/cuda_emu/libtfbs_emu.so (the product's kernel sources on a CUDA-on-host shim)."""
    subprocess.check_call(["make", "-C", EMU, "-j2", "libtfbs_emu.so"], stdout=subprocess.DEVNULL)
    env = dict(os.environ)
    env["TFBS_B200_LIB"] = os.path.join(EMU, "libtfbs_emu.so")
    out = run_marked_gpu_tests(env, "tests/test_large_regions.py", "forced_device_vector")
    assert "5 passed" in out
