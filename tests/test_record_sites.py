"""Binding sites of every record on its own (option "record_sites", tfbs_get_record_sites): per record of the block, the hits of its
region's window patched with that record alone that the unpatched window lacks (change +1) and the reverse (change -1), whoever
carries it, and the flags of the records patch_haplotype would not apply alone.

Checked here:
* every record's flags and sites, in order, against the oracle's patch_haplotype and a NumPy scoring of every complete window
  (test_sites.expected_sites with the one record), on the reference fixture (by hand too), small cohorts, 30-bp PWMs with dense
  indels, an insertion whose bases start several windows at one position, a deletion whose anchor-only windows cancel, a hit whose
  score moves, an always-hit pattern, 32-bit fields, N runs, duplicate BED lines, OtherPattern, records nobody carries (one with a REF
  mismatch, one MNP), records outside the window, a record two regions fetch, same-position records, a block without carriers and a
  block without keys;
* a configuration of exactly one record has that record's sites (also on a configs[2]-shaped block and a 40,000-sample block whose
  fan-out keeps its vectors in device memory);
* bit-identical output across contexts, reseeded repeats, a cold context whose every capacity overflows once, the device-memory
  fan-out, two blocks in flight on two lanes and after the next submit into the slot;
* rows, attribution and sites do not change with the option, the launches it adds, and the calls that must fail;
* the driver's --record_sites file.
The small cases also run on the emulated kernels (tests/cuda_emu) in the CPU suite."""
import os
import subprocess

import numpy as np
import pytest

from find_tfbs_b200 import binding, synth
from find_tfbs_b200.binding import PatternSet
from oracle import pyoracle as ora
import file_writers as fw
import parity_helpers as hp
import test_attribution as ta
import test_sites as ts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "cuda_emu")
MODES = ta.MODES
REC_ARRAYS = ("rec_flags", "site_off", "pattern_index", "start", "score", "change")
REC_LAUNCHES = 8  # what the option adds to a run without option "sites"; with it, none (DESIGN.md, "Record sites")


# ---- running a block ----------------------------------------------------------------------------------------------------------------

def run(ps, blk, mode=binding.ROWS_ALL_KEYS, options=None, record_sites=1):
    """One context: grouped rows (expanded), attribution and sites when the options ask for them, record sites and stats of one block."""
    opts = dict(options or {})
    ctx = binding.Context(0)
    try:
        ctx.set_option("rows_mode", mode)
        ctx.set_option("record_sites", record_sites)
        for k, v in opts.items():
            ctx.set_option(k, v)
        ctx.set_patterns(ps)
        ctx.submit_block(blk)
        g = ta.own(ctx.collect_grouped(expand=True))
        a = ctx.attribution() if opts.get("attribution") else None
        s = ctx.sites() if opts.get("sites") else None
        r = ctx.record_sites() if record_sites else None
        st = ctx.stats()
    finally:
        ctx.close()
    return g, a, s, r, st


def assert_same_records(a, b):
    assert a["n_records"] == b["n_records"]
    for k in REC_ARRAYS:
        assert a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k]), k


# ---- the expectation: patch_haplotype with the one record + every complete window scored in NumPy ------------------------------------

def region_of(blk, v):
    return int(np.searchsorted(blk.var_off, v, side="right")) - 1


def expected_record(ps, blk, v, ref_hits=None):
    """(flags, sorted sites) of record v: OUTSIDE by window membership (var_inwin), REF_MISMATCH / MISSING_CASE from the oracle's
    patch_haplotype panics (-4 / -5)."""
    r = region_of(blk, v)
    pos = int(blk.variants[v]["pos"])
    if not int(blk.region_start[r]) <= pos <= int(blk.region_end[r]):
        return binding.REC_OUTSIDE, []
    try:
        return 0, ts.expected_sites(ps, blk, r, [v], ref_hits)
    except ora.OracleError as e:
        return {-4: binding.REC_REF_MISMATCH, -5: binding.REC_MISSING_CASE}[e.code], []


def check_records(ps, blk, rs, regions=None):
    """Every record (of `regions`, all by default) against expected_record, in order.  Returns the sites checked."""
    n = int(blk.var_off[blk.n_regions])
    assert rs["n_records"] == n and len(rs["rec_flags"]) == n and len(rs["site_off"]) == n + 1 and rs["site_off"][0] == 0
    checked, ref_cache = 0, {}
    for v in range(n):
        r = region_of(blk, v)
        if regions is not None and r not in regions:
            continue
        if r not in ref_cache:
            ref_cache[r] = ts.hit_triples(ps, ts.region_window(blk, r)[1])
        flags, want = expected_record(ps, blk, v, ref_cache[r])
        assert int(rs["rec_flags"][v]) == flags, v
        got = ts.got_sites(rs, v)
        assert got == want, (v, r)
        checked += len(got)
    return checked


def check_single_record_configs(a, s, rs):
    """A configuration of exactly one record has that record's sites.  Returns the configurations compared."""
    coff = a["cfg_rec_off"].astype(np.int64)
    n = 0
    for o in range(int(a["n_cfgs"])):
        if coff[o + 1] - coff[o] == 1:
            v = int(a["cfg_rec"][coff[o]])
            assert rs["rec_flags"][v] == 0 and ts.got_sites(s, o) == ts.got_sites(rs, v), (o, v)
            n += 1
    return n


def check_case(ps, blk, options=None, regions=None):
    """Record sites against the oracle; the same with attribution and sites on, in both row modes, where every one-record configuration
    has its record's sites."""
    g, a, s, rs, st = run(ps, blk, options=options)
    n = check_records(ps, blk, rs, regions)
    for mode in MODES:
        _, a2, s2, rs2, _ = run(ps, blk, mode, dict(options or {}, attribution=1, sites=1))
        assert_same_records(rs, rs2)
        check_single_record_configs(a2, s2, rs2)
    return rs, n


# ---- hand-made cases --------------------------------------------------------------------------------------------------------------

def uncarried_case(carried=True):
    """Region 0: an insertion (carried when `carried`), an SNV nobody carries, a REF mismatch and an MNP nobody carries, a record
    behind the window and two records at one position; region 1 overlaps region 0 and fetches the SNV at 7 too."""
    w = np.array([[100, 0, 0, 0], [0, 100, 0, 0], [5, 7, 11, 13]], np.int32)  # "AC?" scores 200 + the third base's weight
    g = "TTTTTACGTTTTTTTTTTTT"
    blk = hp.hand_block(3, [(0, 19, g), (5, 15, g[5:16])],
                        [(0, 5, "A", "ACTACAC"), (0, 7, "G", "T"), (0, 9, "C", "G"), (0, 12, "TT", "GA"), (0, 25, "T", "A"),
                         (0, 14, "T", "A"), (0, 14, "T", "C"), (1, 7, "G", "T")],
                        [[0, 3], [], [], [], [], [4], [], []] if carried else [[]] * 8)
    ps = PatternSet([{"weights": w, "min_score": 204, "pattern_id": 4}, {"weights": w[::-1, ::-1].copy(), "min_score": 204, "pattern_id": 4, "direction": 1},
                     {"weights": np.array([[0, 0, 0, 50], [50, 0, 0, 0]], np.int32), "min_score": 99, "pattern_id": 9}])
    return ps, blk


# ---- 1 + 2: against the oracle, and the one-record configurations (GPU and emulated kernels) ---------------------------------------------

@pytest.mark.gpu
def test_small_reference_fixture_record_sites():
    ps = ta.acgt_patterns()
    for carriers in ([0], [0, 3, 6], []):
        blk = ta.fixture_block(carriers)
        rs, n = check_case(ps, blk)
        # the SNV A->G at 100 destroys the ACGT window at 100..103, which scores 4000 on both strands, whoever carries it
        assert rs["rec_flags"].tolist() == [0] and ts.got_sites(rs, 0) == [(0, 100, 4000, -1), (1, 100, 4000, -1)]


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2])
def test_small_synthetic_record_sites(seed):
    ps, blk = ta.small_cohort(seed)
    rs, n = check_case(ps, blk)
    assert n > 0 and (rs["change"] > 0).any() and (rs["change"] < 0).any()


@pytest.mark.gpu
def test_small_long_pwms_dense_indels_record_sites():
    ps, blk = ta.long_pwm_dense_indels()
    rs, n = check_case(ps, blk)
    assert n > 0


@pytest.mark.gpu
def test_small_truncation_same_position_record_sites():
    ps, blk = ta.truncation_block()
    rs, n = check_case(ps, blk)
    assert n > 0


@pytest.mark.gpu
def test_small_insertion_deletion_changed_score_record_sites():
    ps, blk = ts.indel_case()
    rs, n = check_case(ps, blk)
    got = [ts.got_sites(rs, v) for v in range(3)]
    # as the one-record configurations of test_sites: the insertion's three AC? windows at its anchor, the deletion's TT hit with the
    # anchor-only TT window cancelled, the SNV's lost / gained pair
    assert got[0] == [(0, 5, 205, 1), (0, 5, 207, 1), (0, 5, 211, -1), (0, 5, 213, 1)]
    assert got[1] == [(1, 12, 207, -1), (2, 10, 100, 1)]
    assert got[2] == [(0, 4, 211, 1), (0, 4, 213, -1)]


@pytest.mark.gpu
def test_small_always_hit_pattern_record_sites():
    ps, blk = ts.always_hit_case()
    rs, n = check_case(ps, blk)
    assert (rs["pattern_index"] == len(ps.items) - 1).sum() > 0


@pytest.mark.gpu
def test_small_scan_format_wide_fields_record_sites():
    ps, blk = ta.small_cohort(1)
    check_case(ps, blk, {"scan_format": 1})


@pytest.mark.gpu
def test_small_two_bed_sets_duplicates_n_runs_other_pattern_record_sites():
    ps, blk = ta.two_beds_n_runs()
    ps = PatternSet(ps.items + [{"kind": binding.PATTERN_OTHER, "pattern_id": 99}])
    blk.inner["multiplicity"] = (np.arange(len(blk.inner)) % 3 + 1).astype(np.uint32)
    rs, n = check_case(ps, blk, regions=set(range(12)))
    assert n > 0


@pytest.mark.gpu
def test_small_uncarried_outside_same_position_two_regions():
    for carried in (True, False):  # False: a block without carriers
        ps, blk = uncarried_case(carried)
        rs, n = check_case(ps, blk)
        R = binding
        assert rs["rec_flags"].tolist() == [0, 0, R.REC_REF_MISMATCH, R.REC_MISSING_CASE, R.REC_OUTSIDE, 0, 0, 0]
        assert all(ts.got_sites(rs, v) == [] for v in (2, 3, 4))
        # the SNV at 7 turns the ACG hit at 5 (211) into ACT (213); region 1 fetches it too and reports it again
        assert ts.got_sites(rs, 1) == ts.got_sites(rs, 7)
        assert {(0, 5, 211, -1), (0, 5, 213, 1)} <= set(ts.got_sites(rs, 1))
        # same position: T->A at 14 gains the TA hit at 13, T->C none
        assert ts.got_sites(rs, 5) == [(2, 13, 100, 1)] and ts.got_sites(rs, 6) == []
    # a REF mismatch some haplotype carries still fails the block, with or without the option
    ps, blk = uncarried_case()
    blk.carriers[2, 0] |= np.uint32(1)
    for opt in (0, 1):
        with pytest.raises(binding.TfbsError) as e:
            run(ps, blk, record_sites=opt)
        assert e.value.code == binding.ERR_REF_MISMATCH


@pytest.mark.gpu
def test_small_block_without_keys_record_sites():
    ps, blk = ta.small_cohort(1)
    b = blk.slice(0, 4)
    b.inner_off[:] = 0
    g, a, s, rs, st = run(ps, b)
    assert st["n_rows"] == 0
    assert check_records(ps, b, rs) > 0


# ---- 3 + 4: determinism, nothing else changes, refusals -----------------------------------------------------------------------------

@pytest.mark.gpu
def test_small_record_sites_deterministic():
    ps, blk = ta.two_beds_n_runs()
    rs = run(ps, blk)[3]
    assert len(rs["change"]) > 1
    for opts in ({}, {"test_reseed": 1}, {"tiny_caps": 1}, {"fan_vector": 1}, {"tiny_caps": 1, "test_reseed": 1, "fan_vector": 1},
                 {"tiny_caps": 1, "attribution": 1, "sites": 1}):
        assert_same_records(rs, run(ps, blk, options=opts)[3])


@pytest.mark.gpu
def test_small_record_sites_dual_stream_and_next_submit():
    ps, b1 = ta.small_cohort(1)
    b2, b3 = ta.small_cohort(2)[1], ta.small_cohort(3)[1]
    want = [run(ps, b, binding.ROWS_VARYING)[3] for b in (b1, b2, b3)]
    for dual in (0, 1):
        ctx = binding.Context(0)
        try:
            ctx.set_option("dual_stream", dual)
            ctx.set_option("record_sites", 1)
            ctx.set_patterns(ps)
            ctx.submit_block(b1)
            ctx.submit_block(b2)
            ctx.collect_grouped()
            ctx.submit_block(b3)  # takes the slot of b1
            assert_same_records(want[0], ctx.record_sites())
            ctx.collect()
            assert_same_records(want[1], ctx.record_sites())
            ctx.collect_grouped()
            assert_same_records(want[2], ctx.record_sites())
        finally:
            ctx.close()


@pytest.mark.gpu
def test_small_record_sites_change_nothing_else_launches_and_refusals():
    ps, blk = ta.small_cohort(2)
    for mode in MODES:
        for opts in ({}, {"attribution": 1}, {"attribution": 1, "sites": 1}):
            g1, a1, s1, _, st1 = run(ps, blk, mode, opts)
            g0, a0, s0, _, st0 = run(ps, blk, mode, opts, record_sites=0)
            for k in g0:
                if isinstance(g0[k], np.ndarray) and k not in ("offset", "packed"):
                    assert np.array_equal(g0[k], g1[k]), k
            assert np.array_equal(ta.rows_packed(g0), ta.rows_packed(g1))
            if a0 is not None:
                ta.assert_same_attribution(a0, a1)
            if s0 is not None:
                ts.assert_same_sites(s0, s1)
            assert st1["scan_launches"] == st0["scan_launches"]
            assert st1["total_launches"] - st0["total_launches"] == (0 if opts.get("sites") else REC_LAUNCHES)
    ctx = binding.Context(0)
    try:
        ctx.set_patterns(ps)
        with pytest.raises(binding.TfbsError) as e:
            ctx.record_sites()
        assert e.value.code == binding.ERR_STATE and "collected" in e.value.message and "record sites" in e.value.message
        ctx.submit_block(blk)
        ctx.collect()
        with pytest.raises(binding.TfbsError) as e:
            ctx.record_sites()
        assert e.value.code == binding.ERR_STATE and "record_sites was off" in e.value.message
        ctx.set_option("record_sites", 1)
        for opt in ("delta", "record_matches"):
            ctx.set_option(opt, 0 if opt == "delta" else 1)
            ctx.submit_block(blk)
            ctx.collect()
            with pytest.raises(binding.TfbsError) as e:
                ctx.record_sites()
            assert e.value.code == binding.ERR_STATE and "full scan" in e.value.message and "record sites" in e.value.message
            ctx.set_option(opt, 1 if opt == "delta" else 0)
        ctx.upload_block(blk)
        ctx.audit()
        ctx.collect()  # the audit leaves a full scan of the block behind
        with pytest.raises(binding.TfbsError) as e:
            ctx.record_sites()
        assert e.value.code == binding.ERR_STATE and "full scan" in e.value.message
        ctx.submit_block(blk)
        ctx.collect()
        assert len(ctx.record_sites()["change"]) > 0
        with pytest.raises(binding.TfbsError) as e:
            ctx.set_option("record_sites", 2)
        assert e.value.code == binding.ERR_INVALID_ARGUMENT and "record_sites must be 0 or 1" in e.value.message
    finally:
        ctx.close()


# ---- 5: the driver ----------------------------------------------------------------------------------------------------------------

RECORD_SITES_HEADER = "#RECORD\tREGION\tPATTERN\tSTRAND\tSTART\tEND\tSCORE\tCHANGE"


def read_record_sites(path):
    lines = open(path).read().splitlines()
    assert lines[0] == RECORD_SITES_HEADER
    out = []
    for ln in lines[1:]:
        f = ln.split("\t")
        assert len(f) == 8 and f[3] in ("+", "-") and f[7] in ("+1", "-1")
        out.append((f[0], f[1], f[2], f[3], int(f[4]), int(f[5]), int(f[6]), int(f[7])))
    return out


def expected_driver_lines(ps, pats, blk):
    """The --record_sites lines of a one-block run: per region, record and site of that record alone that overlaps one of the region's
    inner regions, from the NumPy expectation."""
    out = []
    for r in range(blk.n_regions):
        inner = blk.inner[int(blk.inner_off[r]):int(blk.inner_off[r + 1])]
        region = "%d-%d" % (int(inner["start"].min()), int(inner["end"].max()))  # the merged region
        for v in range(int(blk.var_off[r]), int(blk.var_off[r + 1])):
            flags, sites = expected_record(ps, blk, v)
            if flags:
                continue
            pos, rf, al = ts.record(blk, v)
            for pi, st, sc, ch in sites:
                q = pats[pi]
                L = np.asarray(q["weights"]).reshape(-1, 4).shape[0]
                if not any((int(x["start"]) <= st <= int(x["end"])) or (int(x["start"]) <= st + L - 1 <= int(x["end"])) for x in inner):
                    continue
                out.append(("%d:%s:%s" % (pos + 1, rf, al), region, q["name"], "+" if q["direction"] == 0 else "-", st, st + L - 1, sc, ch))
    return out


@pytest.mark.gpu
def test_small_driver_record_sites(tmp_path):
    """--record_sites on small cohort files (one block, so that region r of the driver is region r of the block) against the NumPy
    expectation; the file is the same with --attribution / --sites, for two --chunk values, and for --devices 0 vs 0,1 where two GPUs
    are present; --audit is refused."""
    pats = synth.make_pwms(4, seed=21, lmin=6, lmax=16)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(16, 24, seed=21, lmax_pattern=lmax, region_len=(80, 400), variant_rate=1 / 10.0, frac_ins=0.15, frac_del=0.15,
                            two_beds=True, same_pos_frac=0.05)
    ps = PatternSet(pats)
    files = fw.cohort_to_files(blk, pats, str(tmp_path / "files"))
    path = str(tmp_path / "rs.tsv")
    p = ta.run_driver(files, str(tmp_path / "out.vcf.gz"), ["--chunk", "10000", "--record_sites", path, "--verbose"])
    assert p.returncode == 0, p.stderr
    assert "Record sites: records without sites" in p.stdout
    got = read_record_sites(path)
    assert len(got) > 0 and got == expected_driver_lines(ps, pats, blk)
    text = open(path).read()
    runs = [["--chunk", "10000", "--attribution", str(tmp_path / "a.tsv"), "--sites", str(tmp_path / "s.tsv")], ["--chunk", "5"], ["--chunk", "3"]]
    try:
        import torch
        if torch.cuda.device_count() >= 2:
            runs.append(["--chunk", "3", "--devices", "0,1"])
    except ImportError:
        pass
    for extra in runs:
        path2 = str(tmp_path / "rs2.tsv")
        p = ta.run_driver(files, str(tmp_path / "out2.vcf.gz"), extra + ["--record_sites", path2])
        assert p.returncode == 0, p.stderr
        assert open(path2).read() == text, extra
    p = ta.run_driver(files, str(tmp_path / "x.vcf.gz"), ["--record_sites", path, "--audit", str(tmp_path / "au.tsv")])
    assert p.returncode != 0 and "--record_sites" in (p.stdout + p.stderr)


def fixture_args(golden_dir, bcf):
    return {"chromosome": "chr1", "bcf": os.path.join(golden_dir, bcf), "reference": os.path.join(golden_dir, "reference_genome.fa"),
            "beds": [os.path.join(golden_dir, "regions1.bed"), os.path.join(golden_dir, "regions2.bed")], "names": ["ACGT"],
            "pwm_file": os.path.join(golden_dir, "pwm_definitions.txt"), "threshold_dir": golden_dir,
            "extra": ["--samples", os.path.join(golden_dir, "samples")]}


@pytest.mark.gpu
def test_small_driver_record_sites_reference_fixture(golden_dir, tmp_path):
    """genotypes2.bcf: the SNV A->G at 100 (1-based 101) destroys the ACGT window at 100..103 scoring 4000 on both strands -- two lines,
    in merged region 100-115.  genotypes.bcf: its one record (POS 1) lies outside every extended window: only the header."""
    out, path = str(tmp_path / "out.vcf.gz"), str(tmp_path / "rs.tsv")
    p = ta.run_driver(fixture_args(golden_dir, "genotypes2.bcf"), out, ["--record_sites", path])
    assert p.returncode == 0, p.stderr
    assert ora.gunzip_file(out) == ora.gunzip_file(os.path.join(golden_dir, "expected_output_2.vcf.gz"))  # the option changes no row
    assert read_record_sites(path) == [("101:A:G", "100-115", "ACGT", "+", 100, 103, 4000, -1), ("101:A:G", "100-115", "ACGT", "-", 100, 103, 4000, -1)]
    p = ta.run_driver(fixture_args(golden_dir, "genotypes.bcf"), out, ["--record_sites", path])
    assert p.returncode == 0, p.stderr
    assert open(path).read() == RECORD_SITES_HEADER + "\n"


# ---- large blocks (GPU only) --------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_configs2_shaped_block_record_sites():
    """A configs[2]-shaped block at 2 % of its regions: one-record configurations against their records everywhere, the records of three
    regions against the oracle."""
    pats, blk = synth.config3(scale=0.02)
    ps = PatternSet(pats)
    g, a, s, rs, st = run(ps, blk, binding.ROWS_VARYING, {"attribution": 1, "sites": 1})
    assert check_single_record_configs(a, s, rs) > 0
    counts = np.bincount(g["region"], minlength=blk.n_regions)
    picks = set(int(r) for r in np.argsort(-counts, kind="stable")[:3])
    assert check_records(ps, blk, rs, picks) > 0


@pytest.mark.gpu
def test_40000_samples_record_sites():
    pats = synth.make_pwms(4, seed=5, lmin=6, lmax=10, pvalue=1e-3)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(40000, 2, seed=5, lmax_pattern=lmax, region_len=(500, 700), variant_rate=1 / 4.0, gap=(100, 300))
    ps = PatternSet(pats)
    g, a, s, rs, st = run(ps, blk, binding.ROWS_VARYING, {"attribution": 1, "sites": 1})
    assert check_single_record_configs(a, s, rs) > 0
    assert check_records(ps, blk, rs, {0}) > 0


# ---- the small cases on the emulated kernels (CPU) ----------------------------------------------------------------------------------

def test_small_cases_on_emulated_kernels():
    """The GPU tests named *small* on tests/cuda_emu/libtfbs_emu.so and the driver linked against it."""
    from test_large_regions import run_marked_gpu_tests
    subprocess.check_call(["make", "-C", EMU, "-j2", "libtfbs_emu.so", "find-tfbs-emu"], stdout=subprocess.DEVNULL)
    env = dict(os.environ, TFBS_B200_LIB=os.path.join(EMU, "libtfbs_emu.so"), TFBS_B200_DRIVER=os.path.join(EMU, "find-tfbs-emu"))
    out = run_marked_gpu_tests(env, "tests/test_record_sites.py", "small")
    assert "16 passed" in out
