"""Binding sites behind the attribution's terms (option "sites", tfbs_get_sites): per configuration, the hits of the region's window
patched with its records alone that the unpatched window lacks (change +1) and the reverse (change -1), as multisets of
(pattern_index, start, score) triples.

Checked here:
* every configuration's sites, in order, against the oracle's patch_haplotype and a NumPy scoring of every complete window, on the
  reference fixture (by hand too), small cohorts, 30-bp PWMs with dense indels, truncations, same-position records and overwrites,
  an insertion whose bases start several windows at one position, a deletion whose anchor-only windows cancel, a hit whose score
  moves, an always-hit pattern, 32-bit fields, N runs, duplicate BED lines, OtherPattern and a block without keys;
* the sites add up to the attribution's terms for every row in both row modes (also on a configs[2]-shaped block and a 40,000-sample
  block whose fan-out keeps its vectors in device memory);
* bit-identical output across contexts, reseeded repeats, a cold context whose every capacity overflows once, the device-memory
  fan-out and two blocks in flight on two lanes, and after the next submit into the slot;
* the rows and the attribution do not change with the option, the launches it adds, and the calls that must fail.
The small cases also run on the emulated kernels (tests/cuda_emu) in the CPU suite."""
import os
import subprocess
from collections import Counter

import numpy as np
import pytest

from find_tfbs_b200 import binding, synth
from find_tfbs_b200.binding import PatternSet
from oracle import pyoracle as ora
import file_writers as fw
import parity_helpers as hp
import test_attribution as ta

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "cuda_emu")
MODES = ta.MODES
SITE_ARRAYS = ("site_off", "pattern_index", "start", "score", "change")
SITE_LAUNCHES = 8  # what the option adds to a run with attribution (DESIGN.md, "Sites")


# ---- running a block ----------------------------------------------------------------------------------------------------------------

def run(ps, blk, mode=binding.ROWS_ALL_KEYS, options=None, sites=1):
    """One context with attribution on: grouped rows (expanded), attribution, sites and stats of one block."""
    ctx = binding.Context(0)
    try:
        ctx.set_option("rows_mode", mode)
        ctx.set_option("attribution", 1)
        ctx.set_option("sites", sites)
        for k, v in (options or {}).items():
            ctx.set_option(k, v)
        ctx.set_patterns(ps)
        ctx.submit_block(blk)
        g = ta.own(ctx.collect_grouped(expand=True))
        a = ctx.attribution()
        s = ctx.sites() if sites else None
        st = ctx.stats()
    finally:
        ctx.close()
    return g, a, s, st


def assert_same_sites(a, b):
    assert a["n_cfgs"] == b["n_cfgs"]
    for k in SITE_ARRAYS:
        assert a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k]), k


# ---- the expected sites: patch_haplotype + every complete window scored in NumPy ------------------------------------------------------

def hit_triples(ps, hap):
    """Multiset of (pattern_index, start, score) of every complete window with score > min_score; N scores 0."""
    out = Counter()
    if not hap:
        return out
    codes = np.array(["ACGTN".index(x.upper()) for x, _ in hap], np.int64)
    pos = np.array([p for _, p in hap], np.int64)
    for pi, item in enumerate(ps.items):
        if item.get("kind", binding.PATTERN_PWM) != binding.PATTERN_PWM:
            continue
        w = np.asarray(item["weights"], np.int64).reshape(-1, 4)
        L = len(w)
        if len(codes) < L:
            continue
        w5 = np.vstack([w.T, np.zeros((1, L), np.int64)])  # [base][column], N = 0
        win = np.lib.stride_tricks.sliding_window_view(codes, L)
        sc = w5[win, np.arange(L)].sum(axis=1)
        for s in np.nonzero(sc > int(item.get("min_score", 0)))[0]:
            out[(pi, int(pos[s]), int(sc[s]))] += 1
    return out


def region_window(blk, r):
    ref = bytes(blk.ref_bases[int(blk.ref_off[r]):int(blk.ref_off[r + 1])]).decode()
    rs = int(blk.region_start[r])
    return (rs, int(blk.region_end[r])), [(c, rs + k) for k, c in enumerate(ref)]


def record(blk, v):
    x = blk.variants[v]
    al = blk.allele_bases
    return (int(x["pos"]), bytes(al[int(x["ref_off"]):int(x["ref_off"]) + int(x["ref_len"])]).decode(),
            bytes(al[int(x["alt_off"]):int(x["alt_off"]) + int(x["alt_len"])]).decode())


def expected_sites(ps, blk, r, records, ref_hits=None):
    """Sorted [(pattern_index, start, score, change)] of the configuration that carries `records` (indices into blk.variants)."""
    rng, ref = region_window(blk, r)
    if ref_hits is None:
        ref_hits = hit_triples(ps, ref)
    hap, _ = ora.patch_haplotype(rng, [record(blk, v) for v in records], ref)
    a = hit_triples(ps, hap)
    out = [k + (1,) for k, n in (a - ref_hits).items() for _ in range(n)] + [k + (-1,) for k, n in (ref_hits - a).items() for _ in range(n)]
    return sorted(out)


def got_sites(s, o):
    lo, hi = int(s["site_off"][o]), int(s["site_off"][o + 1])
    return list(zip(s["pattern_index"][lo:hi].tolist(), s["start"][lo:hi].tolist(), s["score"][lo:hi].tolist(), s["change"][lo:hi].tolist()))


def check_sites(ps, blk, a, s, regions=None):
    """Every configuration of `regions` (all by default) against expected_sites, in order.  Returns the sites checked."""
    assert s["n_cfgs"] == a["n_cfgs"] and len(s["site_off"]) == a["n_cfgs"] + 1 and s["site_off"][0] == 0
    coff = a["cfg_rec_off"].astype(np.int64)
    checked = 0
    ref_cache = {}
    for o in range(int(a["n_cfgs"])):
        r = int(a["cfg_region"][o])
        if regions is not None and r not in regions:
            continue
        if r not in ref_cache:
            ref_cache[r] = hit_triples(ps, region_window(blk, r)[1])
        want = expected_sites(ps, blk, r, a["cfg_rec"][coff[o]:coff[o + 1]].tolist(), ref_cache[r])
        got = got_sites(s, o)
        assert got == want, (o, r)
        checked += len(got)
    return checked


def check_invariant(ps, blk, g, a, s):
    """multiplicity(k) x sum of change over c's sites of the row's pattern_id that overlap inner k == c's term for the row, or 0."""
    pid_of = np.array([int(p["pattern_id"]) for p in ps.items], np.int64)
    len_of = np.array([np.asarray(p["weights"]).reshape(-1, 4).shape[0] if p.get("kind", binding.PATTERN_PWM) == binding.PATTERN_PWM else 0
                       for p in ps.items], np.int64)
    soff = s["site_off"].astype(np.int64)
    owner = np.repeat(np.arange(int(s["n_cfgs"])), np.diff(soff))
    sp_pid, sp_s = pid_of[s["pattern_index"]], s["start"].astype(np.int64)
    sp_e, sp_c = sp_s + len_of[s["pattern_index"]] - 1, s["change"].astype(np.int64)
    toff = a["term_off"].astype(np.int64)
    checked = 0
    for j in range(int(a["n_rows"])):
        r = int(g["region"][j])
        ir = blk.inner[int(g["inner"][j])]
        i_s, i_e, mult = int(ir["start"]), int(ir["end"]), int(ir["multiplicity"])
        sel = (a["cfg_region"][owner] == r) & (sp_pid == int(g["pattern_id"][j])) & (
            ((sp_s >= i_s) & (sp_s <= i_e)) | ((sp_e >= i_s) & (sp_e <= i_e)))  # Range::overlaps, range.rs:18-21
        got = Counter()
        for c, ch in zip(owner[sel].tolist(), sp_c[sel].tolist()):
            got[c] += mult * ch
        got = {c: v for c, v in got.items() if v}
        want = dict(zip(a["term_cfg"][toff[j]:toff[j + 1]].tolist(), a["term_diff"][toff[j]:toff[j + 1]].tolist()))
        assert got == want, j
        checked += len(want)
    return checked


def check_case(ps, blk, options=None, regions=None):
    """Sites against the oracle and the invariant in both row modes; the sites do not depend on the row mode."""
    out = {}
    for mode in MODES:
        g, a, s, st = run(ps, blk, mode, options)
        check_invariant(ps, blk, g, a, s)
        out[mode] = (g, a, s, st)
    assert_same_sites(out[MODES[0]][2], out[MODES[1]][2])
    g, a, s, st = out[binding.ROWS_ALL_KEYS]
    n = check_sites(ps, blk, a, s, regions)
    return g, a, s, st, n


# ---- hand-made cases --------------------------------------------------------------------------------------------------------------

def indel_case():
    """Region 0: an insertion at an A anchor whose bases start several 'AC?' windows at the anchor's position; region 1: a
    deletion whose windows ending on its anchor keep their bases (they cancel); region 2: an SNV that lowers a hit's score but keeps
    it above the threshold (a lost / gained pair)."""
    w = np.array([[100, 0, 0, 0], [0, 100, 0, 0], [5, 7, 11, 13]], np.int32)  # "AC?" scores 200 + the third base's weight
    blk = hp.hand_block(3, [(0, 19, "TTTTTACGTTTTTTTTTTTT"), (0, 19, "TTTTACTTTTTGGGTTTTTT"), (0, 19, "GGGGACTGGGGGGGGGGGGG")],
                        [(0, 5, "A", "ACTACAC"), (1, 10, "TGGG", "T"), (2, 6, "T", "G")],
                        [[0, 3], [1], [0, 2]])
    ps = PatternSet([{"weights": w, "min_score": 204, "pattern_id": 4}, {"weights": w[::-1, ::-1].copy(), "min_score": 204, "pattern_id": 4, "direction": 1},
                     {"weights": np.array([[0, 0, 0, 50], [0, 0, 0, 50]], np.int32), "min_score": 99, "pattern_id": 9}])
    return ps, blk


def always_hit_case():
    """A pattern every window beats (min_score below any score) next to an ordinary one, under insertions and deletions."""
    ps, blk = ta.small_cohort(4)
    items = ps.items + [{"weights": np.array([[1, 2, 3, 4]] * 5, np.int32), "min_score": -1, "pattern_id": 77}]
    return PatternSet(items), blk.slice(0, 6)


# ---- 1 + 2: against the oracle, and the invariant (GPU and emulated kernels) ------------------------------------------------------------

@pytest.mark.gpu
def test_small_reference_fixture_sites():
    ps = ta.acgt_patterns()
    for carriers in ([0], [0, 3, 6]):
        blk = ta.fixture_block(carriers)
        g, a, s, st, n = check_case(ps, blk)
        # the SNV A->G at 100 destroys the ACGT window at 100..103, which scores 4000 on both strands
        assert a["n_cfgs"] == 1 and got_sites(s, 0) == [(0, 100, 4000, -1), (1, 100, 4000, -1)]


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2])
def test_small_synthetic_sites(seed):
    ps, blk = ta.small_cohort(seed)
    g, a, s, st, n = check_case(ps, blk)
    assert n > 0 and (s["change"] > 0).any() and (s["change"] < 0).any()


@pytest.mark.gpu
def test_small_long_pwms_dense_indels_sites():
    ps, blk = ta.long_pwm_dense_indels()
    g, a, s, st, n = check_case(ps, blk)
    assert st["n_truncated"] > 0 and a["cfg_flags"].any() and n > 0


@pytest.mark.gpu
def test_small_truncation_same_position_overwrite_sites():
    ps, blk = ta.truncation_block()
    g, a, s, st, n = check_case(ps, blk)
    assert st["n_truncated"] > 0 and st["n_dropped"] > 0 and n > 0


@pytest.mark.gpu
def test_small_insertion_deletion_changed_score():
    ps, blk = indel_case()
    g, a, s, st, n = check_case(ps, blk)
    by_region = {int(a["cfg_region"][o]): got_sites(s, o) for o in range(int(a["n_cfgs"]))}
    # the inserted ACTACAC starts three AC? windows at the anchor's position, with three scores; the reference's ACG there is lost
    assert by_region[0] == [(0, 5, 205, 1), (0, 5, 207, 1), (0, 5, 211, -1), (0, 5, 213, 1)]
    # the deletion joins T(10) and T(14) into a TT hit and loses the GGT hit at 12; the TT window at 9 that ends on the anchor cancels
    assert by_region[1] == [(1, 12, 207, -1), (2, 10, 100, 1)]
    # the SNV turns the ACT hit at 4 (213) into ACG (211): still a hit, so a lost / gained pair that changes no count
    assert by_region[2] == [(0, 4, 211, 1), (0, 4, 213, -1)]


@pytest.mark.gpu
def test_small_always_hit_pattern():
    ps, blk = always_hit_case()
    g, a, s, st, n = check_case(ps, blk)
    assert (s["pattern_index"] == len(ps.items) - 1).sum() > 0


@pytest.mark.gpu
def test_small_scan_format_wide_fields():
    ps, blk = ta.small_cohort(1)
    check_case(ps, blk, {"scan_format": 1})


@pytest.mark.gpu
def test_small_two_bed_sets_duplicates_n_runs_other_pattern():
    ps, blk = ta.two_beds_n_runs()
    ps = PatternSet(ps.items + [{"kind": binding.PATTERN_OTHER, "pattern_id": 99}])
    blk.inner["multiplicity"] = (np.arange(len(blk.inner)) % 3 + 1).astype(np.uint32)
    g, a, s, st, n = check_case(ps, blk, regions=set(range(12)))
    assert n > 0


@pytest.mark.gpu
def test_small_block_without_keys_sites():
    ps, blk = ta.small_cohort(1)
    b = blk.slice(0, 4)
    b.inner_off[:] = 0
    g, a, s, st = run(ps, b)
    assert a["n_rows"] == 0 and a["n_cfgs"] > 0
    assert check_sites(ps, b, a, s) > 0


# ---- 3 + 4: determinism, nothing else changes, refusals -----------------------------------------------------------------------------

@pytest.mark.gpu
def test_small_sites_deterministic():
    ps, blk = ta.two_beds_n_runs()
    g, a, s, st = run(ps, blk)
    assert len(s["change"]) > 1
    for opts in ({}, {"test_reseed": 1}, {"tiny_caps": 1}, {"fan_vector": 1}, {"tiny_caps": 1, "test_reseed": 1, "fan_vector": 1}):
        assert_same_sites(s, run(ps, blk, options=opts)[2])


@pytest.mark.gpu
def test_small_sites_dual_stream_and_next_submit():
    ps, b1 = ta.small_cohort(1)
    b2, b3 = ta.small_cohort(2)[1], ta.small_cohort(3)[1]
    want = [run(ps, b, binding.ROWS_VARYING)[2] for b in (b1, b2, b3)]
    for dual in (0, 1):
        ctx = binding.Context(0)
        try:
            ctx.set_option("dual_stream", dual)
            ctx.set_option("attribution", 1)
            ctx.set_option("sites", 1)
            ctx.set_patterns(ps)
            ctx.submit_block(b1)
            ctx.submit_block(b2)
            ctx.collect_grouped()
            ctx.submit_block(b3)  # takes the slot of b1
            assert_same_sites(want[0], ctx.sites())
            ctx.collect()
            assert_same_sites(want[1], ctx.sites())
            ctx.collect_grouped()
            assert_same_sites(want[2], ctx.sites())
        finally:
            ctx.close()


@pytest.mark.gpu
def test_small_sites_change_nothing_else_launches_and_refusals():
    ps, blk = ta.small_cohort(2)
    for mode in MODES:
        g1, a1, s1, st1 = run(ps, blk, mode)
        g0, a0, _, st0 = run(ps, blk, mode, sites=0)
        for k in g0:
            if isinstance(g0[k], np.ndarray) and k not in ("offset", "packed"):
                assert np.array_equal(g0[k], g1[k]), k
        assert np.array_equal(ta.rows_packed(g0), ta.rows_packed(g1))
        ta.assert_same_attribution(a0, a1)
        assert st1["total_launches"] - st0["total_launches"] == SITE_LAUNCHES
        st_plain = ta.run(ps, blk, mode, attribution=0)[2]
        assert st0["total_launches"] - st_plain["total_launches"] == ta.LAUNCHES_WITH_KEYS  # sites = 0 adds nothing
    ctx = binding.Context(0)
    try:
        ctx.set_patterns(ps)
        with pytest.raises(binding.TfbsError) as e:
            ctx.sites()
        assert e.value.code == binding.ERR_STATE and "collected" in e.value.message
        ctx.set_option("attribution", 1)
        ctx.submit_block(blk)
        ctx.collect()
        with pytest.raises(binding.TfbsError) as e:
            ctx.sites()
        assert e.value.code == binding.ERR_STATE and "sites was off" in e.value.message
        ctx.set_option("sites", 1)
        for opt in ("delta", "record_matches"):
            ctx.set_option(opt, 0 if opt == "delta" else 1)
            ctx.submit_block(blk)
            ctx.collect()
            with pytest.raises(binding.TfbsError) as e:
                ctx.sites()
            assert e.value.code == binding.ERR_STATE and "full scan" in e.value.message
            ctx.set_option(opt, 1 if opt == "delta" else 0)
        ctx.upload_block(blk)
        ctx.audit()
        ctx.collect()  # the audit leaves a full scan of the block behind
        with pytest.raises(binding.TfbsError) as e:
            ctx.sites()
        assert e.value.code == binding.ERR_STATE and "full scan" in e.value.message
        ctx.set_option("attribution", 0)
        with pytest.raises(binding.TfbsError) as e:
            ctx.submit_block(blk)
        assert e.value.code == binding.ERR_INVALID_ARGUMENT and "needs option attribution" in e.value.message
        ctx.set_option("attribution", 1)
        ctx.submit_block(blk)
        ctx.collect()
        assert len(ctx.sites()["change"]) > 0
        with pytest.raises(binding.TfbsError) as e:
            ctx.set_option("sites", 2)
        assert e.value.code == binding.ERR_INVALID_ARGUMENT and "sites must be 0 or 1" in e.value.message
    finally:
        ctx.close()


# ---- 5: the driver ----------------------------------------------------------------------------------------------------------------

SITES_HEADER = "#ID\tRECORDS\tPATTERN\tSTRAND\tSTART\tEND\tSCORE\tCHANGE"


def read_sites(path):
    lines = open(path).read().splitlines()
    assert lines[0] == SITES_HEADER
    out = []
    for ln in lines[1:]:
        f = ln.split("\t")
        assert len(f) == 8 and f[3] in ("+", "-") and f[7] in ("+1", "-1")
        out.append((f[0], f[1], f[2], f[3], int(f[4]), int(f[5]), int(f[6]), int(f[7])))
    return out


@pytest.mark.gpu
def test_small_driver_sites(tmp_path):
    """--attribution and --sites on the cohort of test_attribution's driver case (one block): per (ID, RECORDS), the sum of CHANGE x
    multiplicity is DIFF; the lines of each term are the NumPy sites of its configuration with the row's pattern_id that overlap the
    row's inner region, in order."""
    pats = synth.make_pwms(4, seed=21, lmin=6, lmax=16)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(16, 24, seed=21, lmax_pattern=lmax, region_len=(80, 400), variant_rate=1 / 10.0, frac_ins=0.15, frac_del=0.15,
                            two_beds=True, same_pos_frac=0.05)
    ps = PatternSet(pats)
    files = fw.cohort_to_files(blk, pats, str(tmp_path / "files"))
    out, apath, spath = str(tmp_path / "out.vcf.gz"), str(tmp_path / "attribution.tsv"), str(tmp_path / "sites.tsv")
    p = ta.run_driver(files, out, ["--chunk", "10000", "--attribution", apath, "--sites", spath])
    assert p.returncode == 0, p.stderr
    att, sites = ta.read_attribution(apath), read_sites(spath)
    ids = ta.vcf_ids(out)
    assert len(ids) > 0 and len(sites) > 0
    # the driver's rows are the oracle's (test_attribution checks that); their region, inner region and pattern by VCF ID
    name = {int(q["pattern_id"]): q["name"] for q in pats if q["direction"] == 0}
    o = hp.run_oracle(ps, blk, binding.ROWS_VARYING)
    rows = {}
    for j in range(len(o["region"])):
        ir = blk.inner[int(o["inner"][j])]
        rid = "regions%d.bed,%s,%d-%d" % (int(ir["bed_index"]) + 1, name[int(o["pattern_id"][j])], int(ir["start"]), int(ir["end"]))
        rows[rid] = (int(o["region"][j]), int(ir["start"]), int(ir["end"]), int(o["pattern_id"][j]))
    # a row's multiplicity: identical lines of its BED file (the files are written from the same peak lists)
    mult = {(int(x["bed_index"]), int(x["start"]), int(x["end"])): int(x["multiplicity"]) for x in blk.inner}
    assert max(mult.values()) > 1
    # groups of lines: (ID, RECORDS) in file order, the same as the attribution file's
    groups = {}
    for x in sites:
        groups.setdefault((x[0], x[1]), []).append(x)
    recs_text = lambda recs: ";".join("%d:%s:%s" % (p + 1, rf, al) for p, rf, al in recs)
    att_keys = [(x["id"], recs_text(x["records"])) for x in att]
    assert list(groups) == att_keys
    for x in att:
        key = (x["id"], recs_text(x["records"]))
        bed = int(x["id"].split(",")[0][len("regions"):-len(".bed")]) - 1
        r, i_s, i_e, pid = rows[x["id"]]
        m = mult[(bed, i_s, i_e)]
        assert sum(g[7] for g in groups[key]) * m == x["diff"], key
        # the NumPy sites of the configuration, restricted to the row's pattern and inner region
        v0, v1 = int(blk.var_off[r]), int(blk.var_off[r + 1])
        recs = [next(v for v in range(v0, v1) if record(blk, v) == rec) for rec in x["records"]]
        want = []
        for pi, st, sc, ch in expected_sites(ps, blk, r, recs):
            q = ps.items[pi]
            L = np.asarray(q["weights"]).reshape(-1, 4).shape[0]
            if int(q["pattern_id"]) != pid or not ((i_s <= st <= i_e) or (i_s <= st + L - 1 <= i_e)):
                continue
            want.append((key[0], key[1], name[pid], "+" if q["direction"] == 0 else "-", st, st + L - 1, sc, ch))
        assert groups[key] == want, key
    # --sites and --audit together are refused
    p = ta.run_driver(files, str(tmp_path / "x.vcf.gz"), ["--sites", spath, "--audit", str(tmp_path / "a.tsv")])
    assert p.returncode != 0 and "--sites" in (p.stdout + p.stderr)


@pytest.mark.gpu
def test_small_driver_sites_reference_fixture(golden_dir, tmp_path):
    """--sites alone on the reference's fixture: the one written row's term is the SNV A->G at 100 (1-based 101), which destroys the ACGT
    window at 100..103 scoring 4000 on both strands -- two lines."""
    args = {"chromosome": "chr1", "bcf": os.path.join(golden_dir, "genotypes2.bcf"), "reference": os.path.join(golden_dir, "reference_genome.fa"),
            "beds": [os.path.join(golden_dir, "regions1.bed"), os.path.join(golden_dir, "regions2.bed")], "names": ["ACGT"],
            "pwm_file": os.path.join(golden_dir, "pwm_definitions.txt"), "threshold_dir": golden_dir,
            "extra": ["--samples", os.path.join(golden_dir, "samples")]}
    out, path = str(tmp_path / "out.vcf.gz"), str(tmp_path / "sites.tsv")
    p = ta.run_driver(args, out, ["--sites", path])
    assert p.returncode == 0, p.stderr
    assert ora.gunzip_file(out) == ora.gunzip_file(os.path.join(golden_dir, "expected_output_2.vcf.gz"))  # the option changes no row
    ids = ta.vcf_ids(out)
    assert len(ids) == 1
    assert read_sites(path) == [(ids[0], "101:A:G", "ACGT", "+", 100, 103, 4000, -1), (ids[0], "101:A:G", "ACGT", "-", 100, 103, 4000, -1)]


# ---- large blocks (GPU only) --------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_configs2_shaped_block_sites():
    """A configs[2]-shaped block at 2 % of its regions: the invariant on every row, the sites of three regions against the oracle."""
    pats, blk = synth.config3(scale=0.02)
    ps = PatternSet(pats)
    g, a, s, st = run(ps, blk, binding.ROWS_VARYING)
    assert check_invariant(ps, blk, g, a, s) > 0
    counts = np.bincount(g["region"], minlength=blk.n_regions)
    picks = set(int(r) for r in np.argsort(-counts, kind="stable")[:3])
    assert check_sites(ps, blk, a, s, picks) > 0


@pytest.mark.gpu
def test_40000_samples_sites():
    pats = synth.make_pwms(4, seed=5, lmin=6, lmax=10, pvalue=1e-3)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(40000, 2, seed=5, lmax_pattern=lmax, region_len=(500, 700), variant_rate=1 / 4.0, gap=(100, 300))
    ps = PatternSet(pats)
    for mode in MODES:
        g, a, s, st = run(ps, blk, mode)
        check_invariant(ps, blk, g, a, s)
    assert check_sites(ps, blk, a, s, {0}) > 0


# ---- the small cases on the emulated kernels (CPU) ----------------------------------------------------------------------------------

def test_small_cases_on_emulated_kernels():
    """The GPU tests named *small* on tests/cuda_emu/libtfbs_emu.so and the driver linked against it."""
    from test_large_regions import run_marked_gpu_tests
    subprocess.check_call(["make", "-C", EMU, "-j2", "libtfbs_emu.so", "find-tfbs-emu"], stdout=subprocess.DEVNULL)
    env = dict(os.environ, TFBS_B200_LIB=os.path.join(EMU, "libtfbs_emu.so"), TFBS_B200_DRIVER=os.path.join(EMU, "find-tfbs-emu"))
    out = run_marked_gpu_tests(env, "tests/test_sites.py", "small")
    assert "15 passed" in out
