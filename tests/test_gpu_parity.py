"""Parity of the CUDA path (through the C ABI) with the CPU oracle: rows, hit lists, haplotype grouping and work counters
must be bit-identical (scores are exact i32 sums, src/pattern.rs:119-151 of the reference; no tolerance applies)."""
import numpy as np
import pytest

from find_tfbs_b200 import binding, synth
from find_tfbs_b200.binding import PatternSet
import parity_helpers as hp

pytestmark = pytest.mark.gpu

ACGT = {"weights": np.eye(4, dtype=np.int32) * 1000, "min_score": 3999, "pattern_id": 0}


def acgt_patterns():
    return PatternSet([dict(ACGT, direction=0), dict(ACGT, direction=1)])


def fixture_block(alt_carriers):
    """The reference's integration fixture (SURVEY App. B): chr1 = 250 x 'A' with ACGT at 100..103, regions1+regions2
    merged, one SNV A->G at 100; 4 samples.  Windows are the merged regions extended by Lmax-1 = 3."""
    genome = bytearray(b"A" * 250)
    genome[100:104] = b"ACGT"
    merged = [(100, 115), (118, 130), (150, 160), (161, 165), (180, 210)]
    bed1 = [(100, 110), (120, 130), (150, 160), (180, 190), (200, 210)]
    bed2 = [(110, 115), (118, 125), (161, 165), (190, 200)]
    regions, inner = [], []
    for m in merged:
        s, e = m[0] - 3, m[1] + 3
        regions.append((s, e, genome[s:e + 1].decode()))
        inner.append([tuple(x) for x in synth.select_inner_peaks(m, [bed1, bed2])])
    return hp.hand_block(4, regions, [(0, 100, "A", "G")], [alt_carriers], inner)


def test_fixture_one_polymorphism():
    """main.rs:559-568 / expected_output_2: INDIVIDUAL1 = 1|0 -> v = [2,4,4,4] for regions1.bed 100-110 only."""
    blk = fixture_block([0])
    g, o = hp.check_parity(acgt_patterns(), blk)
    assert len(g["region"]) == 1
    assert g["region"][0] == 0 and g["pattern_id"][0] == 0
    assert blk.inner[g["inner"][0]]["start"] == 100 and blk.inner[g["inner"][0]]["end"] == 110 and blk.inner[g["inner"][0]]["bed_index"] == 0
    assert (g["left"][0] + g["right"][0]).tolist() == [2, 4, 4, 4]
    assert g["vmin"][0] == 2 and g["vmax"][0] == 4


def test_fixture_no_polymorphism():
    """main.rs:548-557 / expected_output_1: nobody carries the variant -> header only."""
    blk = fixture_block([])
    g, o = hp.check_parity(acgt_patterns(), blk)
    assert len(g["region"]) == 0
    g, o = hp.check_parity(acgt_patterns(), blk, rows_mode=binding.ROWS_ALL_KEYS)
    assert len(g["region"]) == 1 and g["vmin"][0] == 4 and g["vmax"][0] == 4


def test_gataa_strict_threshold_and_n():
    """pattern.rs:285-301: N scores 0, score > min_score is strict."""
    w = np.array([[0, 0, 100, 0], [100, 0, 0, 0], [0, 0, 0, 100], [100, 0, 0, 0], [100, 0, 0, 0]], dtype=np.int32)
    blk = hp.hand_block(1, [(0, 6, "NGATAAN"), (10, 14, "GATAA")], [], [])
    for ms, n in ((499, 2), (500, 0)):
        ps = PatternSet([{"weights": w, "min_score": ms, "pattern_id": 123}])
        g, o = hp.check_parity(ps, blk, rows_mode=binding.ROWS_ALL_KEYS)
        assert len(g["matches"]["start"]) == n


def test_patch_vectors_through_the_kernel():
    """haplotype.rs:172-254 vectors pushed through K1 (the hit list pins every base and position of the patched sequence)."""
    # single-column patterns that hit on one base each: a hit list is then the (nuc, pos) vector of the haplotype
    pats = []
    for b in range(4):
        w = np.zeros((1, 4), dtype=np.int32)
        w[0, b] = 10
        pats.append({"weights": w, "min_score": 5, "pattern_id": b})
    ps = PatternSet(pats)
    ref = "ACGT"
    cases = [
        [(100, "A", "C")], [(1, "C", "N")], [(2, "G", "A")], [(1, "C", "N"), (2, "G", "A")], [(1, "C", "N"), (4, "G", "A")],
        [(1, "C", "NN")], [(2, "G", "NN")], [(3, "T", "NN")], [(1, "CG", "C")], [(2, "GT", "G")], [(0, "AC", "A")],
        [(1, "C", "CTT")], [(1, "C", "TAG"), (2, "G", "T")],
    ]
    regions, variants, carriers = [], [], []
    for i, diffs in enumerate(cases):
        regions.append((1, 2, "CG"))  # window [1,2] of the 4-base genome; haplotype 0 carries the diffs of its case
        for d in diffs:
            variants.append((i, d[0], d[1], d[2]))
            carriers.append([0])
    blk = hp.hand_block(1, regions, variants, carriers)
    hp.check_parity(ps, blk, rows_mode=binding.ROWS_ALL_KEYS)
    assert ref


def test_truncation_and_same_position():
    """haplotype.rs:144-149: a variant overlapped by a previous deletion, or a second variant at one position, truncates."""
    g = "ACGTACGTACGTACGTACGTACGT"
    blk = hp.hand_block(3, [(0, 23, g), (0, 4, g[:5])],
                        [(0, 2, "GTA", "G"), (0, 3, "T", "A"), (0, 10, "G", "A"), (0, 10, "G", "T"), (0, 14, "G", "GAC"),
                         (1, 3, "TA", "T"), (1, 4, "A", "C")],
                        [[0, 1], [0, 2], [3], [3, 4], [1, 5], [0], [0]])
    w = np.array([[1000, 0, 0, 0], [0, 1000, 0, 0]], dtype=np.int32)
    ps = PatternSet([{"weights": w, "min_score": 1500, "pattern_id": 7}, {"weights": w[::-1, ::-1].copy(), "min_score": 1500, "pattern_id": 7, "direction": 1}])
    g_, o = hp.check_parity(ps, blk, rows_mode=binding.ROWS_ALL_KEYS)
    assert o["truncated_regions"] == 2


def test_sequence_keyed_overwrite():
    """haplotype.rs:84 / SURVEY A.6 Q4: two diff lists that patch to the same sequence: the later group is dropped and its
    haplotypes count as reference.  Here hap 1 additionally carries a deletion that starts before the window (not applied)."""
    g = "TTACGTTTTTTT"
    blk = hp.hand_block(2, [(2, 9, g[2:10])], [(0, 1, "TA", "T"), (0, 4, "G", "C")], [[1], [0, 1]])
    w = np.array([[1000, 0, 0, 0], [0, 1000, 0, 0], [0, 0, 1000, 0]], dtype=np.int32)  # ACG
    ps = PatternSet([{"weights": w, "min_score": 2500, "pattern_id": 3}])
    g_, o = hp.check_parity(ps, blk, rows_mode=binding.ROWS_ALL_KEYS)
    assert o["collision_regions"] == 1
    # hap 0 (ACC..) has no hit, hap 1 was dropped into the reference group and so counts the reference hit
    assert (g_["left"][0].tolist(), g_["right"][0].tolist()) == ([0, 1], [1, 1])


def test_errors_match_the_reference_panics():
    w = np.eye(4, dtype=np.int32)
    ps = PatternSet([{"weights": w, "min_score": 0, "pattern_id": 0}])
    cases = [
        (hp.hand_block(1, [(0, 7, "ACGTACGT")], [(0, 2, "A", "T")], [[0]]), binding.ERR_REF_MISMATCH, "doesn't match reference genome"),
        (hp.hand_block(1, [(0, 7, "ACGTACGT")], [(0, 2, "GT", "AC")], [[1]]), binding.ERR_MISSING_CASE, "Missing case in haplotype patcher"),
        (hp.hand_block(1, [(0, 7, "ACGTXCGT")], [], []), binding.ERR_UNKNOWN_NUCLEOTIDE, "Unknown nucleotide"),
        (hp.hand_block(1, [(0, 7, "ACGTACGT")], [(0, 2, "G", "R")], [[]]), binding.ERR_UNKNOWN_NUCLEOTIDE, "Unknown nucleotide"),
    ]
    for blk, code, text in cases:
        with pytest.raises(binding.TfbsError) as e:
            hp.run_gpu(ps, blk)
        assert e.value.code == code and text in e.value.message
        with pytest.raises(hp.ora.OracleError) as e2:
            hp.run_oracle(ps, blk)
        assert e2.value.code == code
    # a mismatching record nobody carries, or one hidden behind a deletion, does not panic in the reference either
    ok = hp.hand_block(1, [(0, 7, "ACGTACGT")], [(0, 2, "A", "T"), (0, 4, "ACG", "A"), (0, 5, "T", "G")], [[], [0], [0]])
    hp.check_parity(ps, ok, rows_mode=binding.ROWS_ALL_KEYS)


def test_empty_and_degenerate_blocks():
    ps = acgt_patterns()
    empty = hp.hand_block(2, [], [], [])
    g = hp.run_gpu(ps, empty)
    assert len(g["region"]) == 0
    # windows shorter than the pattern, an empty reference window, a region without inner regions
    blk = hp.hand_block(2, [(5, 7, "ACG"), (20, 30, ""), (40, 50, "AAACGTACGTA")], [(2, 44, "G", "T")], [[1]],
                        inner=[[(5, 7, 0, 1)], [(20, 30, 0, 1)], []])
    hp.check_parity(ps, blk, rows_mode=binding.ROWS_ALL_KEYS)
    # OtherPattern never matches (pattern.rs:166-168)
    ps2 = PatternSet([dict(ACGT), {"kind": binding.PATTERN_OTHER, "pattern_id": 9}])
    hp.check_parity(ps2, fixture_block([0]), rows_mode=binding.ROWS_ALL_KEYS)


def test_malformed_blocks_are_refused():
    """Argument checks of tfbs_submit_block: a malformed block is an error (never an out-of-bounds access on the device), the
    context stays usable and a failed submit leaves no block behind."""
    ps = acgt_patterns()
    good = fixture_block([0])
    ctx = binding.Context(0)
    ctx.set_patterns(ps)

    def refused(mutate, text):
        blk = fixture_block([0])
        mutate(blk)
        with pytest.raises(binding.TfbsError) as e:
            ctx.submit_block(blk)
        assert e.value.code == binding.ERR_INVALID_ARGUMENT and text in e.value.message, e.value.message
        with pytest.raises(binding.TfbsError) as e2:  # nothing to collect, nothing resident
            ctx.run_resident()
        assert e2.value.code == binding.ERR_STATE

    def set_variant(field, value):
        def f(blk):
            blk.variants[0][field] = value
        return f

    refused(set_variant("alt_len", 0), "empty allele")
    refused(set_variant("ref_off", 10 ** 6), "outside allele_bases")
    refused(set_variant("carrier_row", 77), "no carrier row")

    def bad_window(blk):
        blk.region_end[1] = blk.region_start[1] - 1
    refused(bad_window, "invalid extended window")

    def bad_offsets(blk):
        blk.var_off[2] = 5
        blk.var_off[3] = 1
    refused(bad_offsets, "non-decreasing")

    def long_ref(blk):
        blk.ref_off[1:] += 100
    refused(long_ref, "longer than the region")
    ctx.submit_block(good)
    hp.assert_rows_equal(ctx.collect(), hp.run_oracle(ps, good))
    ctx.close()


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_synthetic_small(seed):
    pats = synth.make_pwms(6, seed=seed, lmin=4, lmax=30)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(12, 40, seed=seed, lmax_pattern=lmax, region_len=(50, 600), variant_rate=1 / 20.0)
    hp.check_parity(PatternSet(pats), blk)
    hp.check_parity(PatternSet(pats), blk, rows_mode=binding.ROWS_ALL_KEYS, matches=False)


def test_synthetic_two_beds_n_runs_lowercase_same_pos():
    pats = synth.make_pwms(8, seed=11, lmin=6, lmax=24)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(20, 60, seed=11, lmax_pattern=lmax, region_len=(80, 700), variant_rate=1 / 12.0, frac_ins=0.15, frac_del=0.15,
                            n_runs=12, lowercase_frac=0.1, two_beds=True, same_pos_frac=0.08)
    g, o = hp.check_parity(PatternSet(pats), blk, rows_mode=binding.ROWS_ALL_KEYS)
    assert o["truncated_regions"] > 0


def test_config5_long_pwm_dense_variants():
    """BASELINE.json configs[4]: 30-bp PWMs, dense rare variants, >= 30% indels, overlapping / same-position records, N runs;
    every window with score == min_score must NOT be a hit (strict >): the oracle enumerates hits, equality of the lists is the audit."""
    pats = synth.make_pwms(5, seed=5, lmin=30, lmax=30, pvalue=1e-3)
    blk = synth.make_cohort(30, 30, seed=5, lmax_pattern=30, region_len=(100, 500), variant_rate=1 / 8.0, frac_ins=0.2, frac_del=0.2,
                            n_runs=4, same_pos_frac=0.1)
    hp.check_parity(PatternSet(pats), blk, rows_mode=binding.ROWS_ALL_KEYS)


def test_threshold_boundary_ties():
    """A pattern whose min_score equals an attainable score: windows scoring exactly min_score are not hits, min_score-1 makes them hits."""
    rng = np.random.default_rng(3)
    w = rng.integers(-3, 4, size=(8, 4)).astype(np.int32) * 100
    blk = synth.make_cohort(6, 20, seed=9, lmax_pattern=8, region_len=(200, 400))
    best = int(w.max(axis=1).sum())
    counts = []
    for ms in (best - 401, best - 400, best - 301, best - 300):
        ps = PatternSet([{"weights": w, "min_score": ms, "pattern_id": 1}])
        g, o = hp.check_parity(ps, blk, rows_mode=binding.ROWS_ALL_KEYS)
        counts.append(o["n_hits"])
    assert counts[0] >= counts[1] >= counts[2] >= counts[3] and counts[0] > counts[3]


def tie_patterns_and_block():
    """Patterns with coarse weights (many attainable ties) and a cohort with dense indels, overwrites and truncations."""
    rng = np.random.default_rng(3)
    w = rng.integers(-3, 4, size=(8, 4)).astype(np.int32) * 100
    best = int(w.max(axis=1).sum())
    pats = [{"weights": w, "min_score": best - 400, "pattern_id": 1, "direction": 0},
            {"weights": w[::-1, ::-1].copy(), "min_score": best - 400, "pattern_id": 1, "direction": 1}]
    pats += synth.make_pwms(2, seed=77, lmin=6, lmax=14)
    for p in pats[2:]:
        p["pattern_id"] += 2
    blk = synth.make_cohort(12, 24, seed=13, lmax_pattern=14, region_len=(100, 500), variant_rate=1 / 10.0, frac_ins=0.15, frac_del=0.2,
                            same_pos_frac=0.1, n_runs=3, two_beds=True)
    return PatternSet(pats), blk


def test_audit_enumerates_ties_and_flags():
    """tfbs_audit_block: the windows scoring exactly min_score (strict >, pattern.rs:151) and the truncated / overwritten haplotypes
    (haplotype.rs:144-149, :84) are the same sets the oracle finds; the context is left with a normal run of the block."""
    ps, blk = tie_patterns_and_block()
    oa = hp.oracle_audit(ps, blk)
    au, rows, st = hp.gpu_audit(ps, blk)
    assert not au["truncated"]
    assert len(oa["ties"]) > 0 and au["ties"] == oa["ties"]
    assert np.array_equal(au["hap_flags"], oa["hap_flags"])
    assert (au["hap_flags"] & binding.HAP_TRUNCATED).any()
    hp.assert_rows_equal(rows, hp.run_oracle(ps, blk))
    assert st["n_hits"] == oa["n_hits"]
    # a match buffer that is too small is enlarged by the audit itself
    au_small, _, _ = hp.gpu_audit(ps, blk, {"max_matches": 50})
    assert not au_small["truncated"] and au_small["ties"] == oa["ties"]
    # a fixture without any tie: ACGT scores 4000 against min_score 3999, the next best window scores 3000
    au2, _, _ = hp.gpu_audit(acgt_patterns(), fixture_block([0]))
    assert len(au2["ties"]) == 0 and not au2["hap_flags"].any()
    # min_score 4000 makes the perfect ACGT windows ties instead of hits: 7 reference-carrying haplotypes share group 0, one window per strand
    tie_ps = PatternSet([dict(ACGT, min_score=4000, direction=0), dict(ACGT, min_score=4000, direction=1)])
    au3, rows3, _ = hp.gpu_audit(tie_ps, fixture_block([0]))
    assert au3["ties"] == {(0, 0, -1, 100), (0, 1, -1, 100)} and len(rows3["region"]) == 0


def test_wide_fields_and_forced_format():
    """Weights too large for the 21-bit packed fields use the two-32-bit-field tables; results must not change."""
    pats = synth.make_pwms(4, seed=21, lmin=10, lmax=20)
    for p in pats:
        p["weights"] = (p["weights"].astype(np.int64) * 40).astype(np.int32)
        p["min_score"] = int(p["min_score"]) * 40
    blk = synth.make_cohort(8, 25, seed=21, lmax_pattern=20, region_len=(100, 500))
    hp.check_parity(PatternSet(pats), blk, rows_mode=binding.ROWS_ALL_KEYS)
    pats2 = synth.make_pwms(4, seed=22, lmin=10, lmax=20)
    a = hp.run_gpu(PatternSet(pats2), blk, rows_mode=binding.ROWS_ALL_KEYS, options={"scan_format": 1})
    b = hp.run_gpu(PatternSet(pats2), blk, rows_mode=binding.ROWS_ALL_KEYS)
    hp.assert_rows_equal(a, b)
    # always-hit and never-hit thresholds
    pats3 = synth.make_pwms(2, seed=23, lmin=5, lmax=9)
    pats3[0]["min_score"] = pats3[1]["min_score"] = -10 ** 9
    pats3[2]["min_score"] = pats3[3]["min_score"] = 10 ** 9
    hp.check_parity(PatternSet(pats3), synth.make_cohort(3, 6, seed=2, lmax_pattern=9, region_len=(30, 90)), rows_mode=binding.ROWS_ALL_KEYS)


def test_pattern_chunks_and_region_batches():
    """Small shared-memory budget -> several pattern chunks; small scratch budget -> several region batches."""
    pats = synth.make_pwms(30, seed=31, lmin=8, lmax=30)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(10, 80, seed=31, lmax_pattern=lmax, region_len=(100, 400), two_beds=True)
    ps = PatternSet(pats)
    base = hp.run_oracle(ps, blk, binding.ROWS_ALL_KEYS, True)
    for opts in ({"table_budget_kb": 16}, {"scratch_mb": 64}, {"table_budget_kb": 24, "scratch_mb": 64, "scan_ctas_per_sm": 1}):
        g = hp.run_gpu(ps, blk, binding.ROWS_ALL_KEYS, True, opts)
        hp.assert_rows_equal(g, base)
        hp.assert_matches_equal(g, base)


def test_resident_path_and_rerun():
    pats = synth.make_pwms(5, seed=41)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(16, 30, seed=41, lmax_pattern=lmax, region_len=(100, 900))
    ps = PatternSet(pats)
    o = hp.run_oracle(ps, blk)
    ctx = binding.Context(0)
    ctx.set_patterns(ps)
    ctx.upload_block(blk)
    for _ in range(3):  # idempotent: same rows every run
        ctx.run_resident()
        hp.assert_rows_equal(ctx.collect(), o)
    ctx.submit_block(blk)
    hp.assert_rows_equal(ctx.collect(), o)
    ctx.close()


def test_many_samples_few_groups():
    """Carriers drawn from founder classes: thousands of haplotypes collapse into a few groups per region (SURVEY D3)."""
    pats = synth.make_pwms(4, seed=51, lmin=8, lmax=16)
    blk = synth.make_cohort(700, 12, seed=51, lmax_pattern=16, region_len=(200, 600), ld_blocks=12)
    g, o = hp.check_parity(PatternSet(pats), blk)
    assert o["n_groups"] < 12 * 14


def test_config4_biobank_shape():
    """BASELINE.json configs[3] in shape: tens of thousands of haplotypes per region (here 40,000), few regions, founder classes so
    that the oracle stays fast; exercises the per-region loops over H and the wide carrier rows.  Sample-block sharding of the same
    block must concatenate to the same rows."""
    from find_tfbs_b200 import sharding
    pats = synth.make_pwms(3, seed=51, lmin=8, lmax=16, pvalue=3e-3)
    ps = PatternSet(pats)
    blk = synth.make_cohort(20000, 4, seed=52, lmax_pattern=16, region_len=(200, 400), ld_blocks=40)
    g, o = hp.check_parity(ps, blk, rows_mode=binding.ROWS_ALL_KEYS, matches=False)
    assert g["left"].shape[1] == 20000 and len(g["region"]) > 0
    parts = [hp.run_gpu(ps, sharding.sample_block(blk, s0, s1), rows_mode=binding.ROWS_ALL_KEYS) for s0, s1 in ((0, 7000), (7000, 20000))]
    merged = sharding.merge_sample_shards(parts)  # applies the min != max filter after the gather
    hp.assert_rows_equal(merged, hp.run_oracle(ps, blk, binding.ROWS_VARYING))


def test_config4_dense_sample_blocks():
    """BASELINE.json configs[3] as generated for the bench (synth.config4: a record every ~4 bp, 1/k spectrum, uniform carriers, so
    nearly every haplotype of a region is distinct and one cluster spans the region), in sample blocks: grouped rows of every block in
    ALL_KEYS mode, merged by tfbs_merge_sample_blocks (min != max over all samples after the gather), equal to the oracle run block
    by block and merged in Python -- and to the oracle on the whole cohort where no sequence-keyed overwrite happened (SURVEY A.6 Q4:
    the winner is chosen per block)."""
    from find_tfbs_b200 import sharding
    pats, blk = synth.config4(n_regions=3, n_samples=208, seed=14, n_pwms=4)
    ps = PatternSet(pats)
    cuts = ((0, 80), (80, 160), (160, 208))
    ctx = binding.Context(0)
    try:
        ctx.set_option("rows_mode", binding.ROWS_ALL_KEYS)
        ctx.set_patterns(ps)
        parts, dropped = [], 0
        for a, b in cuts:
            ctx.submit_block(sharding.sample_block(blk, a, b))
            parts.append(binding.own_grouped(ctx.collect_grouped()))
            dropped += ctx.stats()["n_dropped"]
    finally:
        ctx.close()
    merged = binding.merge_sample_blocks(parts)
    o_parts = [hp.run_oracle(ps, sharding.sample_block(blk, a, b), binding.ROWS_ALL_KEYS) for a, b in cuts]
    hp.assert_rows_equal(merged, sharding.merge_sample_shards(o_parts))
    assert len(merged["region"]) > 0
    if dropped == 0:
        hp.assert_rows_equal(merged, hp.run_oracle(ps, blk, binding.ROWS_VARYING))


def test_config2_slice_properties():
    """configs[1] at 3% size against the oracle, plus size-independent properties of the rows."""
    pats, blk = synth.config2(scale=0.03)
    ps = PatternSet(pats)
    g, o = hp.check_parity(ps, blk, matches=False)
    v = g["left"].astype(np.int64) + g["right"]
    assert np.array_equal(v.min(axis=1), g["vmin"]) and np.array_equal(v.max(axis=1), g["vmax"])
    assert np.all(g["vmin"] != g["vmax"])
    key = g["region"].astype(np.int64) * (1 << 32) + g["pattern_id"].astype(np.int64) * (1 << 16)
    assert np.all(np.diff(g["region"].astype(np.int64)) >= 0)
    assert np.all(np.diff(key) >= 0)
    # splitting the block into two halves of regions gives the same rows (regions are independent, main.rs:395-429)
    h = blk.n_regions // 2
    a = hp.run_gpu(ps, blk.slice(0, h))
    b = hp.run_gpu(ps, blk.slice(h, blk.n_regions))
    assert len(a["region"]) + len(b["region"]) == len(g["region"])
    assert np.array_equal(np.concatenate([a["left"], b["left"]]), g["left"])
    assert np.array_equal(np.concatenate([a["region"], b["region"] + h]), g["region"])


def test_config2_full_size_properties():
    """BASELINE.json configs[1] at FULL size (100 samples x 10,000 regions x 50 PWMs, both strands): the two scan modes (every distinct
    haplotype scored in full / configurations) must agree row for row and counter for counter, row min / max and ordering must be
    consistent, and EVERY region of the block must equal the oracle's rows (about a hundred seconds of CPU on the box's cores)."""
    import os
    scale = float(os.environ.get("TFBS_TEST_SCALE", "1.0"))  # the emulated run of this file uses a small fraction
    pats, blk = synth.config2(scale=scale)
    ps = PatternSet(pats)
    d = hp.run_gpu(ps, blk, options={"rows_width": 0})
    f = hp.run_gpu(ps, blk, options={"delta": 0})
    hp.assert_rows_equal(d, f)
    for k in ("executed_cells", "nominal_cells", "n_hits", "n_groups", "n_rows", "n_dropped", "n_truncated"):
        assert d["stats"][k] == f["stats"][k], k
    assert f["stats"]["evaluated_cells"] == f["stats"]["executed_cells"] > d["stats"]["evaluated_cells"] > 0
    assert d["count_bytes"] == 1 and f["count_bytes"] == 4
    v = d["left"].astype(np.int64) + d["right"]
    assert np.array_equal(v.min(axis=1), d["vmin"]) and np.array_equal(v.max(axis=1), d["vmax"]) and np.all(d["vmin"] != d["vmax"])
    key = d["region"].astype(np.int64) * (1 << 32) + d["pattern_id"].astype(np.int64) * (1 << 16)
    assert np.all(np.diff(key) >= 0)
    o = hp.run_oracle(ps, blk, 0, False, os.cpu_count() or 4, 50)  # the whole block, chunks of 50 regions like main.rs:378
    hp.assert_rows_equal(d, o)
    hp.check_stats(d["stats"], o)


def test_config3_full_size_random_regions_vs_oracle():
    """BASELINE.json configs[2] at FULL size (the bench workload: 2,504 samples x 4,873 merged regions x 401 PWMs on both strands) in one
    block through the default path, rows collected GROUPED and expanded on the host: 56 regions in four random places must equal the
    oracle's rows (the oracle needs about half a minute of one core per region), min / max / ordering must be consistent everywhere."""
    import os
    pats, blk = synth.config3(scale=float(os.environ.get("TFBS_TEST_SCALE", "1.0")))
    ps = PatternSet(pats)
    ctx = binding.Context(0)
    try:
        ctx.set_patterns(ps)
        ctx.submit_block(blk)
        g = ctx.collect_grouped()
        st = ctx.stats()
        assert g["n_rows"] == st["n_rows"] > 0 and g["bytes"] < 0.4e9  # the rows of the whole chromosome cross PCIe in well under 0.4 GB
        key = g["region"].astype(np.int64) * (1 << 32) + g["pattern_id"].astype(np.int64) * (1 << 16)
        assert np.all(np.diff(key) >= 0) and np.all(g["vmin"] != g["vmax"])
        rng = np.random.default_rng(7)
        picked = 0
        for r0 in sorted(int(x) for x in rng.integers(0, max(1, blk.n_regions - 14), size=4)):
            r1 = min(blk.n_regions, r0 + 14)
            picked += r1 - r0
            o = hp.run_oracle(ps, blk.slice(r0, r1), 0, False, os.cpu_count() or 4, 1)
            rows = np.nonzero((g["region"] >= r0) & (g["region"] < r1))[0]
            assert len(rows) == len(o["region"]) and len(rows) > 0
            first, n = int(rows[0]), len(rows)
            assert np.array_equal(rows, np.arange(first, first + n))
            left = np.zeros((n, blk.n_samples), dtype=np.uint32)
            right = np.zeros((n, blk.n_samples), dtype=np.uint32)
            import ctypes as C
            assert binding.lib().tfbs_expand_rows(C.byref(g["_c"]), first, n, left.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                  right.ctypes.data_as(C.POINTER(C.c_uint32))) == 0
            assert np.array_equal(g["region"][rows] - r0, o["region"]) and np.array_equal(g["pattern_id"][rows], o["pattern_id"])
            assert np.array_equal(g["inner"][rows] - int(blk.inner_off[r0]), o["inner"])
            assert np.array_equal(g["vmin"][rows], o["vmin"]) and np.array_equal(g["vmax"][rows], o["vmax"])
            assert np.array_equal(left, o["left"]) and np.array_equal(right, o["right"])
            v = left.astype(np.int64) + right
            assert np.array_equal(v.min(axis=1), o["vmin"]) and np.array_equal(v.max(axis=1), o["vmax"])
        assert picked >= 50
    finally:
        ctx.close()


def test_region_sharding_on_device():
    """The multi-GPU partition (find_tfbs_b200/sharding.py) run shard by shard on one device equals the unsharded rows."""
    from find_tfbs_b200 import sharding
    pats = synth.make_pwms(6, seed=61, lmin=8, lmax=20)
    blk = synth.make_cohort(10, 50, seed=61, lmax_pattern=20, region_len=(100, 500), two_beds=True)
    ps = PatternSet(pats)
    full = hp.run_gpu(ps, blk)
    for world in (2, 4):
        parts, offs = [], []
        for rank in range(world):
            shard, r0, i0 = sharding.shard_block(blk, world, rank, lmax=20)
            assert shard.carriers.shape[0] <= max(1, len(shard.variants))  # compact: only the carrier rows the shard uses
            parts.append(hp.run_gpu(ps, shard))
            offs.append((r0, i0))
        hp.assert_rows_equal(sharding.merge_rows(parts, offs), full)


def test_sample_block_sharding_on_device():
    """configs[3] semantics at small scale: sample blocks are scored independently (ALL_KEYS rows), concatenated along the sample
    axis and filtered for min != max after the gather (main.rs:450-458 needs every sample)."""
    from find_tfbs_b200 import sharding
    pats = synth.make_pwms(5, seed=71, lmin=8, lmax=18)
    blk = synth.make_cohort(24, 30, seed=71, lmax_pattern=18, region_len=(100, 400), frac_del=0.0, variant_rate=1 / 25.0)
    ps = PatternSet(pats)
    o = hp.run_oracle(ps, blk)
    assert o["collision_regions"] == 0
    full = hp.run_gpu(ps, blk)
    hp.assert_rows_equal(full, o)
    parts = [hp.run_gpu(ps, sharding.sample_block(blk, a, b), rows_mode=binding.ROWS_ALL_KEYS) for a, b in ((0, 7), (7, 16), (16, 24))]
    hp.assert_rows_equal(sharding.merge_sample_shards(parts), full)


def test_config3_like_many_samples_many_pwms():
    """configs[2] shape at reduced size: 2,504 samples, several hundred patterns (several shared-memory table chunks), two BED sets.
    Oracle parity on a few regions; size-independent properties on more."""
    pats = synth.make_pwms(150, seed=81, lmin=8, lmax=24)
    lmax = max(p["weights"].shape[0] for p in pats)
    ps = PatternSet(pats)
    for kw in ({"ld_blocks": 40, "two_beds": True}, {"variant_rate": 1 / 60.0}):  # few groups per region / nearly every haplotype distinct
        blk = synth.make_cohort(2504, 4, seed=81, lmax_pattern=lmax, region_len=(150, 300), **kw)
        o = hp.run_oracle(ps, blk, 0, False, 16, 1)
        g = hp.run_gpu(ps, blk)
        hp.assert_rows_equal(g, o)
        hp.check_stats(g["stats"], o)
        assert g["stats"]["scan_launches"] >= 2  # more than one pattern chunk
    big = synth.make_cohort(2504, 40, seed=82, lmax_pattern=lmax, region_len=(200, 1200), two_beds=True)
    a = hp.run_gpu(ps, big)
    b = hp.run_gpu(ps, big, options={"delta": 0, "scratch_mb": 2048})
    hp.assert_rows_equal(a, b)
    v = a["left"].astype(np.int64) + a["right"]
    assert np.array_equal(v.min(axis=1), a["vmin"]) and np.array_equal(v.max(axis=1), a["vmax"]) and np.all(a["vmin"] != a["vmax"])


def test_delta_scoring_corner_cases():
    """Delta scoring paths the other tests do not reach: several pattern chunks, several region batches, the fall-back to a full scan
    when the reference-hit buffer overflows, long regions (several tiles / plane rounds per sequence) and 32-column patterns."""
    pats = synth.make_pwms(30, seed=31, lmin=8, lmax=30)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(10, 80, seed=31, lmax_pattern=lmax, region_len=(100, 400), two_beds=True)
    ps = PatternSet(pats)
    base = hp.run_oracle(ps, blk, binding.ROWS_ALL_KEYS, False)
    for opts in ({"table_budget_kb": 16}, {"scratch_mb": 64}, {"refhit_cap": 3}, {"table_budget_kb": 24, "scratch_mb": 64, "refhit_cap": 50}):
        g = hp.run_gpu(ps, blk, binding.ROWS_ALL_KEYS, False, opts)
        hp.assert_rows_equal(g, base)
        hp.check_stats(g["stats"], base)
    # long regions and the longest supported patterns
    pats = synth.make_pwms(3, seed=32, lmin=31, lmax=32) + synth.make_pwms(2, seed=33, lmin=1, lmax=3)
    for i, p in enumerate(pats):
        p["pattern_id"] = i // 2
    blk = synth.make_cohort(6, 4, seed=32, lmax_pattern=32, region_len=(2500, 4200), variant_rate=1 / 40.0, frac_ins=0.1, frac_del=0.1)
    hp.check_parity(PatternSet(pats), blk, rows_mode=binding.ROWS_ALL_KEYS)


def test_narrow_row_counts():
    """Option rows_width = 0: counts come back as u8 / u16 / u32, whichever holds the largest count of the block; values are unchanged.
    Large counts are forced with duplicate BED lines (the multiplicity of an inner region, SURVEY A.6 Q3)."""
    pats = synth.make_pwms(6, seed=91, lmin=6, lmax=16, pvalue=1e-2)
    ps = PatternSet(pats)
    for mult, width in ((1, 1), (300, 2), (70000, 4)):
        blk = synth.make_cohort(9, 25, seed=91, lmax_pattern=16, region_len=(150, 500))
        blk.inner["multiplicity"] = mult
        o = hp.run_oracle(ps, blk) if mult == 1 else None
        base = hp.run_gpu(ps, blk)
        assert base["count_bytes"] == 4
        if o is not None:
            hp.assert_rows_equal(base, o)
        for opts in ({"rows_width": 0}, {"rows_width": 0, "scratch_mb": 64}):
            g = hp.run_gpu(ps, blk, options=opts)
            assert g["count_bytes"] == width, (g["count_bytes"], int(base["vmax"].max()))
            hp.assert_rows_equal(g, base)


def test_grouped_rows_two_blocks_in_flight_and_scratch_growth():
    """The default path end to end: (i) started with minimal scratch (option tiny_caps) every capacity overflows once and the block is
    repeated until it fits -- same rows; (ii) two blocks in flight on one context (a third submit is refused), rows collected in
    submission order as GROUPED rows (one count per distinct haplotype + the haplotype -> group map per region) and expanded on the
    host by tfbs_expand_rows -- equal to the oracle's (left, right) vectors; (iii) two resident runs in flight, one collected dense
    (expanded on the device), one grouped."""
    for seed in (1, 2, 3):
        pats = synth.make_pwms(6, seed=seed)
        lmax = max(p["weights"].shape[0] for p in pats)
        blk = synth.make_cohort(12, 10, seed=seed, lmax_pattern=lmax, region_len=(200, 600), two_beds=True, n_runs=2, same_pos_frac=0.1,
                                frac_ins=0.15, frac_del=0.15)
        ps = PatternSet(pats)
        for mode in (binding.ROWS_VARYING, binding.ROWS_ALL_KEYS):
            o = hp.run_oracle(ps, blk, mode, False)
            d = hp.run_gpu(ps, blk, mode, False, {"tiny_caps": 1})
            hp.assert_rows_equal(d, o)
            hp.check_stats(d["stats"], o)
            for dual in (0, 1):  # option dual_stream: slot 1 runs on a second lane (own streams and scratch)
                ctx = binding.Context(0)
                try:
                    ctx.set_option("rows_mode", mode)
                    ctx.set_patterns(ps)
                    ctx.set_option("dual_stream", dual)
                    half = blk.n_regions // 2
                    b1, b2 = blk.slice(0, half), blk.slice(half, blk.n_regions)
                    ctx.submit_block(b1)
                    ctx.submit_block(b2)
                    with pytest.raises(binding.TfbsError) as e:
                        ctx.submit_block(b1)
                    assert e.value.code == binding.ERR_STATE
                    g1 = ctx.collect_grouped(expand=True)
                    g1 = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in g1.items()}
                    g2 = ctx.collect_grouped(expand=True)
                    hp.assert_rows_equal(g1, hp.run_oracle(ps, b1, mode, False))
                    hp.assert_rows_equal(g2, hp.run_oracle(ps, b2, mode, False))
                    assert set(np.unique(g2["bits"]).tolist()) <= {0, 1, 2, 4, 8, 16, 32}
                    ctx.upload_block(blk)
                    ctx.run_resident()
                    ctx.run_resident()
                    hp.assert_rows_equal(ctx.collect(), o)
                    hp.assert_rows_equal(ctx.collect_grouped(expand=True), o)
                    with pytest.raises(binding.TfbsError):
                        ctx.collect()  # nothing in flight any more
                    if dual:  # result arena: the block of slot 0 (lane 0) writes the first half, that of slot 1 (lane 1) the second
                        raw = np.zeros((4 << 20) + 64, dtype=np.uint8)
                        arena = raw[(-raw.ctypes.data) % 64:][:4 << 20]  # 64-byte aligned
                        ctx.set_result_arena(arena)
                        for b in (b1, b2, b1):
                            ctx.submit_block(b)
                            ctx.collect_grouped()
                        h0, h1 = binding.read_arena(arena, 0, expand=True), binding.read_arena(arena, 1, expand=True)
                        assert h0["sequence"] == 2 and h1["sequence"] == 1
                        hp.assert_rows_equal(h0, hp.run_oracle(ps, b1, mode, False))
                        hp.assert_rows_equal(h1, hp.run_oracle(ps, b2, mode, False))
                        ctx.set_result_arena(None)
                        assert ctx.stats()["n_regions"] == b1.n_regions
                finally:
                    ctx.close()


def test_dual_stream_set_after_upload():
    """Option dual_stream set after tfbs_upload_block: two runs of the resident block in flight, one on each lane, both read the
    one copy of the block on the device and return the oracle's rows."""
    pats = synth.make_pwms(5, seed=43)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(12, 10, seed=43, lmax_pattern=lmax, region_len=(100, 600), frac_ins=0.15, frac_del=0.15)
    ps = PatternSet(pats)
    o = hp.run_oracle(ps, blk)
    ctx = binding.Context(0)
    try:
        ctx.set_patterns(ps)
        ctx.upload_block(blk)
        ctx.set_option("dual_stream", 1)
        ctx.run_resident()
        ctx.run_resident()
        hp.assert_rows_equal(ctx.collect(), o)
        hp.assert_rows_equal(ctx.collect(), o)
    finally:
        ctx.close()


def test_dual_stream_audit_takes_the_last_block():
    """With dual_stream on, tfbs_audit_block audits the block most recently submitted, whichever lane ran it: after b1 and b2 (of
    different region counts) are collected, the audit is that of b2 -- the same ties and flags as a single-stream context's audit of
    b2 -- and the normal run it leaves behind returns b2's rows."""
    ps, blk = tie_patterns_and_block()
    b1, b2 = blk.slice(0, 16), blk.slice(16, blk.n_regions)
    ref, _, _ = hp.gpu_audit(ps, b2)
    assert len(ref["region"]) > 0
    ctx = binding.Context(0)
    try:
        ctx.set_patterns(ps)
        ctx.set_option("dual_stream", 1)
        ctx.submit_block(b1)
        ctx.submit_block(b2)
        ctx.collect()
        ctx.collect()
        au = ctx.audit()
        assert len(au["hap_group"]) == b2.n_regions * 2 * b2.n_samples  # tfbs_audit.n_regions is b2's
        for k in ("region", "pattern_index", "group", "start", "hap_group", "hap_flags"):
            assert np.array_equal(au[k], ref[k]), k
        hp.assert_rows_equal(ctx.collect(), hp.run_oracle(ps, b2))
    finally:
        ctx.close()


def test_bed_merge_on_device():
    """tfbs_merge_regions == load_peak_files' merge (bed.rs:37-45, range.rs:43-87): the reference's own vector (bed.rs:67-95), random
    range sets against the literal fold (synth.merge_regions), ties in start, touching and nested ranges, sizes around the tile."""
    ctx = binding.Context(0)
    try:
        ref = [(100, 110), (120, 130), (150, 160), (180, 190), (200, 210), (110, 115), (118, 125), (161, 165), (190, 200)]
        assert ctx.merge_regions(ref) == [(100, 115), (118, 130), (150, 160), (161, 165), (180, 210)]
        assert ctx.merge_regions([]) == [] and ctx.merge_regions([(5, 5)]) == [(5, 5)]
        assert ctx.merge_regions([(0, 0), (0, 0), (1, 1)]) == [(0, 0), (1, 1)]  # equal ranges join, start = end + 1 does not (inclusive ends)
        rng = np.random.default_rng(7)
        for n, span, width in ((2, 10, 5), (255, 3000, 20), (256, 3000, 20), (257, 1000, 3), (700, 200000, 400), (5000, 10 ** 7, 3000), (3000, 500, 50)):
            s = rng.integers(0, span, size=n)
            e = s + rng.integers(0, width, size=n)
            ranges = list(zip(s.tolist(), e.tolist()))
            assert ctx.merge_regions(ranges) == synth.merge_regions(ranges), n
        with pytest.raises(binding.TfbsError):
            ctx.merge_regions([(10, 5), (1, 2)])
    finally:
        ctx.close()


def test_repeat_with_another_seed():
    """A hash collision (signature, configuration or sequence hash) repeats the block with another seed; option test_reseed makes the
    first attempt of every block count as one: the rows of the repeated run equal the oracle's, sequence-keyed overwrites included."""
    pats = synth.make_pwms(4, seed=77, lmin=8, lmax=14, pvalue=2e-3)
    blk = synth.make_cohort(30, 10, seed=77, lmax_pattern=14, region_len=(80, 400), variant_rate=0.08, frac_del=0.2, same_pos_frac=0.1)
    ps = PatternSet(pats)
    g = hp.run_gpu(ps, blk, options={"test_reseed": 1})
    hp.assert_rows_equal(g, hp.run_oracle(ps, blk, 0))
    assert g["stats"]["n_dropped"] == hp.run_gpu(ps, blk)["stats"]["n_dropped"]
