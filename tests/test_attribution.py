"""Attribution of the result rows (option "attribution", tfbs_get_attribution): per row, the configurations -- the records of one
cluster of nearby records that a haplotype carries together -- whose count difference to the region's reference haplotype is not 0.

Checked here:
* the invariant, against the oracle: for every row, haplotype and sample, the count is ref_count + the terms whose configuration the
  haplotype's group lists, exactly, in both row modes, on the reference fixture, small cohorts, 30-bp PWMs with dense indels
  (truncations, same-position records, overwritten haplotypes), duplicate BED lines, two BED sets with N runs, OtherPattern, a block
  without keys, a configs[2]-shaped block (on a few of its regions) and a 40,000-sample block whose fan-out keeps its vectors in
  device memory;
* every term on its own: a configuration's difference is the oracle's count on the reference window patched with its records alone,
  minus the reference window's count (one block per region, sample i's left haplotype carries configuration i);
* bit-identical output across contexts, reseeded repeats, a cold context whose every capacity overflows once, the device-memory
  fan-out and two blocks in flight on two streams;
* the rows do not change with the option, the launches it adds, and the calls that must fail;
* the driver's --attribution file against the VCF and the oracle.
The small cases and the driver case also run on the emulated kernels (tests/cuda_emu) in the CPU suite."""
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

from find_tfbs_b200 import binding, synth
from find_tfbs_b200.binding import Block, PatternSet
from oracle import pyoracle as ora
import file_writers as fw
import parity_helpers as hp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "cuda_emu")
DRIVER = os.environ.get("TFBS_B200_DRIVER") or os.path.join(ROOT, "find_tfbs_b200", "find-tfbs-b200")
MODES = (binding.ROWS_VARYING, binding.ROWS_ALL_KEYS)
ARRAYS = ("ref_count", "term_off", "term_cfg", "term_diff", "cfg_region", "cfg_flags", "cfg_rec_off", "cfg_rec", "group_cfg_off", "group_cfg")
LAUNCHES_WITH_KEYS, LAUNCHES_WITHOUT_KEYS = 10, 6  # what the option adds to a run (DESIGN.md, "Attribution")
ACGT = {"weights": np.eye(4, dtype=np.int32) * 1000, "min_score": 3999, "pattern_id": 0}


# ---- running a block --------------------------------------------------------------------------------------------------------------

def own(g):
    return {k: (np.array(v, copy=True) if isinstance(v, np.ndarray) else v) for k, v in g.items() if k != "_c"}


def run(ps, blk, mode, options=None, attribution=1):
    """One context: grouped rows (expanded), the attribution and the stats of one block."""
    ctx = binding.Context(0)
    try:
        ctx.set_option("rows_mode", mode)
        ctx.set_option("attribution", attribution)
        for k, v in (options or {}).items():
            ctx.set_option(k, v)
        ctx.set_patterns(ps)
        ctx.submit_block(blk)
        g = own(ctx.collect_grouped(expand=True))
        a = ctx.attribution() if attribution else None
        st = ctx.stats()
    finally:
        ctx.close()
    return g, a, st


def rows_packed(g):
    """The packed words of the grouped rows in row order."""
    words = (g["n_groups"][g["region"]].astype(np.int64) * g["bits"].astype(np.int64) + 31) // 32
    first = np.repeat(g["offset"].astype(np.int64), words)
    return g["packed"][first + np.arange(int(words.sum())) - np.repeat(np.cumsum(words) - words, words)]


def assert_same_attribution(a, b):
    assert a["n_rows"] == b["n_rows"] and a["n_cfgs"] == b["n_cfgs"] and a["n_groups_total"] == b["n_groups_total"]
    for k in ARRAYS:
        assert a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k]), k


# ---- the invariant ----------------------------------------------------------------------------------------------------------------

def check_structure(g, a):
    n, nc = int(a["n_rows"]), int(a["n_cfgs"])
    assert n == len(g["region"])
    gbase = np.concatenate([[0], np.cumsum(g["n_groups"].astype(np.int64))])
    assert a["n_groups_total"] == gbase[-1]
    toff, coff, goff = (a[k].astype(np.int64) for k in ("term_off", "cfg_rec_off", "group_cfg_off"))
    assert toff[0] == 0 and np.all(np.diff(toff) >= 0) and coff[0] == 0 and np.all(np.diff(coff) >= 1) and goff[0] == 0
    # terms: non-zero, in ascending configuration id, configurations of the row's region
    row_of = np.repeat(np.arange(n), np.diff(toff))
    assert np.all(a["term_diff"] != 0)
    assert np.array_equal(a["cfg_region"][a["term_cfg"]], g["region"][row_of])
    same = row_of[1:] == row_of[:-1]
    assert np.all(np.diff(a["term_cfg"].astype(np.int64))[same] > 0)
    # configurations are numbered by region; their records are records of that region, in position order
    assert np.all(np.diff(a["cfg_region"].astype(np.int64)) >= 0)
    if nc:
        owner = np.repeat(np.arange(nc), np.diff(coff))
        r = a["cfg_region"][owner]
        assert np.all(a["cfg_rec"] >= g["var_off"][r]) and np.all(a["cfg_rec"] < g["var_off"][r + 1])
        pos = g["var_pos"][a["cfg_rec"]]
        assert np.all(np.diff(pos)[owner[1:] == owner[:-1]] >= 0)
    # group lists: nothing for the reference haplotype, configurations of the group's region
    R = len(g["n_groups"])
    if R and gbase[-1]:
        firsts = gbase[:-1][g["n_groups"] > 0]
        assert np.all(goff[firsts + 1] == goff[firsts])
        gowner = np.repeat(np.arange(gbase[-1]), np.diff(goff))
        greg = np.repeat(np.arange(R), g["n_groups"].astype(np.int64))
        assert np.array_equal(a["cfg_region"][a["group_cfg"]], greg[gowner])


def counts_from_attribution(g, a):
    """(left, right) of every row rebuilt as ref_count + the terms whose configuration the haplotype's group lists."""
    n, nc, S = int(a["n_rows"]), int(a["n_cfgs"]), int(g["n_samples"])
    gbase = np.concatenate([[0], np.cumsum(g["n_groups"].astype(np.int64))])
    M = sp.csr_matrix((np.ones(len(a["group_cfg"]), np.int64), a["group_cfg"].astype(np.int64), a["group_cfg_off"].astype(np.int64)),
                      shape=(int(gbase[-1]), nc))
    T = sp.csr_matrix((a["term_diff"].astype(np.int64), a["term_cfg"].astype(np.int64), a["term_off"].astype(np.int64)), shape=(n, nc))
    left, right = np.zeros((n, S), np.int64), np.zeros((n, S), np.int64)
    hg = g["hap_group"].astype(np.int64)
    for r in np.unique(g["region"]):
        rows = np.nonzero(g["region"] == r)[0]
        V = (M[gbase[r]:gbase[r + 1]] @ T[rows].T).toarray()  # groups x rows
        base = a["ref_count"][rows].astype(np.int64)[:, None]
        left[rows] = base + V[hg[r, 0::2]].T
        right[rows] = base + V[hg[r, 1::2]].T
    return left, right


def with_block_arrays(g, blk):
    g["var_off"], g["var_pos"] = blk.var_off.astype(np.int64), blk.variants["pos"]
    return g


def check_invariant(ps, blk, modes=MODES, options=None, oracle=None):
    """Rows equal the oracle's, and the attribution rebuilds every sample's (left, right) of every row exactly."""
    out = {}
    for mode in modes:
        o = oracle[mode] if oracle else hp.run_oracle(ps, blk, mode)
        g, a, st = run(ps, blk, mode, options)
        hp.assert_rows_equal(g, o)
        check_structure(with_block_arrays(g, blk), a)
        left, right = counts_from_attribution(g, a)
        assert np.array_equal(left, o["left"].astype(np.int64)) and np.array_equal(right, o["right"].astype(np.int64))
        out[mode] = (g, a, st, o)
    return out


# ---- every term on its own --------------------------------------------------------------------------------------------------------

def region_configs_block(blk, r, configs):
    """One region of blk; sample i's left haplotype carries the records configs[i] (indices into blk.variants), the right ones nothing."""
    used = sorted(set(v for c in configs for v in c))
    row = {v: k for k, v in enumerate(used)}
    S = max(1, len(configs))
    pitch = max(1, (2 * S + 31) // 32)
    car = np.zeros((max(1, len(used)), pitch), np.uint32)
    for i, c in enumerate(configs):
        for v in c:
            car[row[v], (2 * i) // 32] |= np.uint32(1 << ((2 * i) % 32))
    var = blk.variants[used].copy() if used else np.zeros(0, binding.VARIANT_DTYPE)
    var["carrier_row"] = np.arange(len(used), dtype=np.uint32)
    ro, io = blk.ref_off, blk.inner_off
    return Block(S, blk.region_start[r:r + 1], blk.region_end[r:r + 1], np.array([0, ro[r + 1] - ro[r]], np.uint64),
                 blk.ref_bases[int(ro[r]):int(ro[r + 1])], np.array([0, io[r + 1] - io[r]], np.uint32), blk.inner[int(io[r]):int(io[r + 1])],
                 np.array([0, len(used)], np.uint32), var, blk.allele_bases, car)


def oracle_config_diffs(ps, blk, r, configs):
    """Per configuration {(inner index in the region, pattern_id): count with the records alone - reference count} and the reference
    counts {(inner, pattern_id): count}; a configuration whose haplotype the oracle overwrote is run again in a block of its own."""
    o = hp.run_oracle(ps, region_configs_block(blk, r, configs), binding.ROWS_ALL_KEYS, True)  # (hap_flags come with the hit list)
    diffs = [dict() for _ in configs]
    ref = {}
    for j in range(len(o["region"])):
        key = (int(o["inner"][j]), int(o["pattern_id"][j]))
        ref[key] = int(o["right"][j][0])
        for i in range(len(configs)):
            d = int(o["left"][j][i]) - int(o["right"][j][i])
            if d:
                diffs[i][key] = d
    flags = o["hap_flags"].reshape(-1)
    for i in range(len(configs)):
        if len(configs) > 1 and flags[2 * i] & binding.HAP_OVERWRITTEN:
            diffs[i] = oracle_config_diffs(ps, blk, r, [configs[i]])[0][0]
    return diffs, ref


def check_terms(ps, blk, g, a, regions=None):
    """Every term and every reference count of the rows of `regions` (all with rows by default) against oracle_config_diffs."""
    coff = a["cfg_rec_off"].astype(np.int64)
    toff = a["term_off"].astype(np.int64)
    checked = 0
    for r in (np.unique(g["region"]) if regions is None else regions):
        ids = np.nonzero(a["cfg_region"] == r)[0]
        rows = np.nonzero(g["region"] == r)[0]
        if not len(rows):
            continue
        configs = [a["cfg_rec"][coff[o]:coff[o + 1]].tolist() for o in ids]
        diffs, ref = oracle_config_diffs(ps, blk, int(r), configs)
        for j in rows:
            key = (int(g["inner"][j]) - int(blk.inner_off[r]), int(g["pattern_id"][j]))
            want = {int(o): diffs[k][key] for k, o in enumerate(ids) if key in diffs[k]}
            got = dict(zip(a["term_cfg"][toff[j]:toff[j + 1]].tolist(), a["term_diff"][toff[j]:toff[j + 1]].tolist()))
            assert got == want, (int(r), key)
            assert int(a["ref_count"][j]) == ref.get(key, 0)
            checked += len(got)
    return checked


# ---- cases ------------------------------------------------------------------------------------------------------------------------

def acgt_patterns():
    return PatternSet([dict(ACGT, direction=0), dict(ACGT, direction=1)])


def fixture_block(alt_carriers):
    """The reference's integration fixture: 250 x 'A' with ACGT at 100..103, regions1 + regions2 merged, one SNV A->G at 100."""
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


def small_cohort(seed):
    pats = synth.make_pwms(6, seed=seed, lmin=4, lmax=30)
    lmax = max(p["weights"].shape[0] for p in pats)
    return PatternSet(pats), synth.make_cohort(12, 40, seed=seed, lmax_pattern=lmax, region_len=(50, 600), variant_rate=1 / 20.0)


def long_pwm_dense_indels():
    """configs[4]-style: 30-bp PWMs, dense records with 40 % indels, same-position records, N runs."""
    pats = synth.make_pwms(5, seed=5, lmin=30, lmax=30, pvalue=1e-3)
    blk = synth.make_cohort(30, 30, seed=5, lmax_pattern=30, region_len=(100, 500), variant_rate=1 / 8.0, frac_ins=0.2, frac_del=0.2,
                            n_runs=4, same_pos_frac=0.1)
    return PatternSet(pats), blk


def truncation_block():
    """Truncations (a record inside a deletion, two records at one position) and a sequence-keyed overwrite, by hand."""
    g = "ACGTACGTACGTACGTACGTACGT"
    blk = hp.hand_block(4, [(0, 23, g), (0, 4, g[:5]), (2, 9, "ACGTTTTT")],
                        [(0, 2, "GTA", "G"), (0, 3, "T", "A"), (0, 10, "G", "A"), (0, 10, "G", "T"), (0, 14, "G", "GAC"),
                         (1, 3, "TA", "T"), (1, 4, "A", "C"), (2, 1, "TA", "T"), (2, 4, "G", "C")],
                        [[0, 1], [0, 2], [3], [3, 4], [1, 5], [0], [0], [1], [0, 1]])
    w = np.array([[1000, 0, 0, 0], [0, 1000, 0, 0]], dtype=np.int32)
    ps = PatternSet([{"weights": w, "min_score": 1500, "pattern_id": 7}, {"weights": w[::-1, ::-1].copy(), "min_score": 1500, "pattern_id": 7, "direction": 1},
                     {"weights": np.array([[1000, 0, 0, 0], [0, 1000, 0, 0], [0, 0, 1000, 0]], np.int32), "min_score": 2500, "pattern_id": 3}])
    return ps, blk


def two_beds_n_runs():
    pats = synth.make_pwms(8, seed=11, lmin=6, lmax=24)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(20, 60, seed=11, lmax_pattern=lmax, region_len=(80, 700), variant_rate=1 / 12.0, frac_ins=0.15, frac_del=0.15,
                            n_runs=12, lowercase_frac=0.1, two_beds=True, same_pos_frac=0.08)
    return PatternSet(pats), blk


# ---- 1 + 2: the invariant and every term, small cases (GPU and emulated kernels) ----------------------------------------------------

@pytest.mark.gpu
def test_small_reference_fixture():
    for carriers in ([0], [0, 3, 6], []):
        out = check_invariant(acgt_patterns(), fixture_block(carriers))
        g, a = out[binding.ROWS_ALL_KEYS][:2]
        check_terms(acgt_patterns(), fixture_block(carriers), g, a)
    g, a = check_invariant(acgt_patterns(), fixture_block([0]))[binding.ROWS_VARYING][:2]
    # INDIVIDUAL1 = 1|0: the SNV destroys both ACGT hits of regions1.bed 100-110 (main.rs:559-568)
    assert a["n_rows"] == 1 and a["ref_count"].tolist() == [2] and a["term_diff"].tolist() == [-2]
    assert a["cfg_rec"].tolist() == [0] and a["n_cfgs"] == 1 and not a["cfg_flags"].any()


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2])
def test_small_synthetic(seed):
    ps, blk = small_cohort(seed)
    out = check_invariant(ps, blk)
    g, a = out[binding.ROWS_ALL_KEYS][:2]
    assert a["n_rows"] > 0 and len(a["term_cfg"]) > 0
    assert check_terms(ps, blk, g, a) > 0


@pytest.mark.gpu
def test_small_long_pwms_dense_indels():
    ps, blk = long_pwm_dense_indels()
    out = check_invariant(ps, blk)
    g, a, st, o = out[binding.ROWS_ALL_KEYS]
    assert st["n_truncated"] > 0 and a["cfg_flags"].any()  # configurations that run into the truncation exit
    assert check_terms(ps, blk, g, a) > 0


@pytest.mark.gpu
def test_small_truncation_same_position_overwrite():
    ps, blk = truncation_block()
    out = check_invariant(ps, blk)
    g, a, st, o = out[binding.ROWS_ALL_KEYS]
    assert st["n_truncated"] > 0 and st["n_dropped"] > 0 and a["cfg_flags"].any()
    check_terms(ps, blk, g, a)


@pytest.mark.gpu
def test_small_duplicate_bed_lines():
    ps, blk = small_cohort(3)
    blk.inner["multiplicity"] = (np.arange(len(blk.inner)) % 3 + 1).astype(np.uint32)  # the C struct points at these arrays
    out = check_invariant(ps, blk)
    g, a = out[binding.ROWS_ALL_KEYS][:2]
    check_terms(ps, blk, g, a)


@pytest.mark.gpu
def test_small_two_bed_sets_n_runs_other_pattern():
    ps, blk = two_beds_n_runs()
    ps = PatternSet(ps.items + [{"kind": binding.PATTERN_OTHER, "pattern_id": 99}])
    out = check_invariant(ps, blk)
    g, a = out[binding.ROWS_ALL_KEYS][:2]
    assert check_terms(ps, blk, g, a, regions=np.unique(g["region"])[:12]) > 0


@pytest.mark.gpu
def test_small_block_without_keys():
    """No inner region, so no key: no rows and no terms, but the configurations and group lists are there."""
    ps, blk = small_cohort(1)
    b2 = hp.hand_block(3, [(0, 11, "ACGTACGTACGT")], [(0, 2, "G", "A"), (0, 5, "C", "T")], [[0, 1], [2]], inner=[[]])
    for b in (b2, blk.slice(0, 4)):
        if b is not b2:
            b.inner_off[:] = 0  # every region loses its inner regions
        g, a, st = run(ps, b, binding.ROWS_ALL_KEYS)
        g0, _, st0 = run(ps, b, binding.ROWS_ALL_KEYS, attribution=0)
        assert a["n_rows"] == 0 and len(a["term_cfg"]) == 0 and a["term_off"].tolist() == [0] and a["n_cfgs"] > 0
        assert a["n_groups_total"] == int(g["n_groups"].sum()) and len(a["group_cfg"]) > 0
        assert st["total_launches"] - st0["total_launches"] == LAUNCHES_WITHOUT_KEYS


# ---- 3 + 4: determinism, repeats, nothing changes -----------------------------------------------------------------------------------

@pytest.mark.gpu
def test_small_deterministic_across_contexts_repeats_and_fanout():
    ps, blk = two_beds_n_runs()
    for mode in MODES:
        g, a, st = run(ps, blk, mode)
        assert len(a["term_cfg"]) > 1 and a["n_cfgs"] > 1
        for opts in ({}, {"test_reseed": 1}, {"tiny_caps": 1}, {"fan_vector": 1}, {"tiny_caps": 1, "test_reseed": 1, "fan_vector": 1}):
            g2, a2, _ = run(ps, blk, mode, opts)
            assert_same_attribution(a, a2)
            for k in ("region", "inner", "pattern_id", "vmin", "vmax", "left", "right", "hap_group", "n_groups"):
                assert np.array_equal(g[k], g2[k]), (opts, k)


@pytest.mark.gpu
def test_small_two_blocks_in_flight_dual_stream():
    """Blocks alternate between the two lanes, two in flight: each block's attribution equals the one of a context of its own."""
    ps, b1 = small_cohort(1)
    b2 = small_cohort(2)[1]
    want = [run(ps, b, binding.ROWS_VARYING)[1] for b in (b1, b2, b1)]
    ctx = binding.Context(0)
    try:
        ctx.set_option("dual_stream", 1)
        ctx.set_option("attribution", 1)
        ctx.set_patterns(ps)
        got = []
        ctx.submit_block(b1)
        ctx.submit_block(b2)
        got.append((own(ctx.collect_grouped()), ctx.attribution()))
        ctx.submit_block(b1)
        got.append((ctx.collect(), ctx.attribution()))
        got.append((own(ctx.collect_grouped()), ctx.attribution()))
        # a full scan (always on lane 0) after blocks on both lanes: refused, not the older attribution
        ctx.set_option("delta", 0)
        ctx.submit_block(b2)
        ctx.collect()
        with pytest.raises(binding.TfbsError) as e:
            ctx.attribution()
        assert e.value.code == binding.ERR_STATE and "full scan" in e.value.message
    finally:
        ctx.close()
    for w, (rows, a) in zip(want, got):
        assert a["n_rows"] == len(rows["region"])
        assert_same_attribution(w, a)


@pytest.mark.gpu
def test_small_attribution_survives_the_next_submit():
    """Two blocks in flight on one context: collect A, submit C into A's slot, then ask for the attribution: A's comes back, whole,
    while C runs; then B's and C's after their collects."""
    ps, b_a = small_cohort(1)
    b_b, b_c = small_cohort(2)[1], small_cohort(3)[1]
    want = [run(ps, b, binding.ROWS_VARYING)[1] for b in (b_a, b_b, b_c)]
    assert want[0]["n_rows"] != want[2]["n_rows"] or len(want[0]["term_cfg"]) != len(want[2]["term_cfg"])
    for resident in (False, True):
        ctx = binding.Context(0)
        try:
            ctx.set_option("attribution", 1)
            ctx.set_patterns(ps)
            ctx.submit_block(b_a)
            ctx.submit_block(b_b)
            g = own(ctx.collect_grouped())
            ctx.submit_block(b_c)  # takes the slot of A
            a = ctx.attribution()
            assert a["n_rows"] == len(g["region"])
            assert_same_attribution(want[0], a)
            rows = ctx.collect()
            assert_same_attribution(want[1], ctx.attribution())
            assert ctx.attribution()["n_rows"] == len(rows["region"])
            if resident:  # and a run that reuses B's slot before B's attribution is read
                ctx.upload_block(b_c)  # (drops C, which is in flight)
                ctx.run_resident()
                ctx.run_resident()
                ctx.collect_grouped()
                ctx.run_resident()
                assert_same_attribution(want[2], ctx.attribution())
                ctx.collect_grouped()
            else:
                ctx.collect_grouped()
            assert_same_attribution(want[2], ctx.attribution())
        finally:
            ctx.close()


@pytest.mark.gpu
def test_small_rows_unchanged_launches_and_refusals():
    ps, blk = small_cohort(2)
    for mode in MODES:
        g1, a, st1 = run(ps, blk, mode)
        g0, _, st0 = run(ps, blk, mode, attribution=0)
        for k in g0:  # (the packed payload's order in `packed` is not fixed, the rows are: compared through left / right and rows_packed)
            if isinstance(g0[k], np.ndarray) and k not in ("offset", "packed"):
                assert np.array_equal(g0[k], g1[k]), k
        assert np.array_equal(rows_packed(g0), rows_packed(g1))
        assert st1["total_launches"] - st0["total_launches"] == LAUNCHES_WITH_KEYS
        d1 = hp.run_gpu(ps, blk, mode, options={"attribution": 1})
        d0 = hp.run_gpu(ps, blk, mode)
        hp.assert_rows_equal(d1, d0)
    ctx = binding.Context(0)
    try:
        ctx.set_patterns(ps)
        with pytest.raises(binding.TfbsError) as e:
            ctx.attribution()  # nothing collected yet
        assert e.value.code == binding.ERR_STATE and "collected" in e.value.message
        ctx.submit_block(blk)
        ctx.collect()
        with pytest.raises(binding.TfbsError) as e:
            ctx.attribution()  # option off
        assert e.value.code == binding.ERR_STATE and "attribution was off" in e.value.message
        ctx.set_option("attribution", 1)
        for opt in ("delta", "record_matches"):
            ctx.set_option(opt, 0 if opt == "delta" else 1)
            ctx.submit_block(blk)
            ctx.collect()
            with pytest.raises(binding.TfbsError) as e:
                ctx.attribution()
            assert e.value.code == binding.ERR_STATE and "full scan" in e.value.message
            ctx.set_option(opt, 1 if opt == "delta" else 0)
        ctx.submit_block(blk)
        ctx.collect()
        assert ctx.attribution()["n_rows"] > 0
        with pytest.raises(binding.TfbsError):
            ctx.set_option("attribution", 2)
    finally:
        ctx.close()


# ---- 5: the driver ------------------------------------------------------------------------------------------------------------------

def run_driver(args, out, extra):
    cmd = [DRIVER, "--chromosome", args["chromosome"], "--input", args["bcf"], "--output", out, "--reference", args["reference"],
           "--bed", ",".join(args["beds"]), "--pwm_names", ",".join(args["names"]), "--pwm_file", args["pwm_file"],
           "--pwm_threshold_directory", args["threshold_dir"], "--pwm_threshold", "0.0001"] + args.get("extra", []) + extra
    return subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)


def read_attribution(path):
    lines = open(path).read().splitlines()
    assert lines[0] == "#ID\tREF_COUNT\tRECORDS\tDIFF\tHAPLOTYPES\tTRUNCATES"
    out = []
    for ln in lines[1:]:
        f = ln.split("\t")
        assert len(f) == 6 and f[5] in ("0", "1")
        recs = [(int(p) - 1, rf, al) for p, rf, al in (x.split(":") for x in f[2].split(";"))]
        out.append({"id": f[0], "ref": int(f[1]), "records": recs, "diff": int(f[3]), "haps": int(f[4]), "trunc": int(f[5])})
    return out


def vcf_ids(path):
    return [ln.split("\t")[2] for ln in ora.gunzip_file(path).splitlines() if ln and not ln.startswith("#")]


def check_driver_file(att, ids):
    """The attribution's IDs are the VCF's row IDs in the VCF's order, every row has at least one line."""
    seen = []
    for x in att:
        if not seen or seen[-1] != x["id"]:
            seen.append(x["id"])
    assert seen == ids and len(set(ids)) == len(ids)


@pytest.mark.gpu
def test_small_driver_attribution(tmp_path):
    pats = synth.make_pwms(4, seed=21, lmin=6, lmax=16)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(16, 24, seed=21, lmax_pattern=lmax, region_len=(80, 400), variant_rate=1 / 10.0, frac_ins=0.15, frac_del=0.15,
                            two_beds=True, same_pos_frac=0.05)
    ps = PatternSet(pats)
    files = fw.cohort_to_files(blk, pats, str(tmp_path / "files"))
    out, path = str(tmp_path / "out.vcf.gz"), str(tmp_path / "attribution.tsv")
    p = run_driver(files, out, ["--chunk", "10000", "--attribution", path])  # one block: region r of the driver is region r of blk
    assert p.returncode == 0, p.stderr
    att = read_attribution(path)
    ids = vcf_ids(out)
    assert len(ids) > 0
    check_driver_file(att, ids)
    # the oracle's rows under their VCF IDs
    name = {int(q["pattern_id"]): q["name"] for q in pats if q["direction"] == 0}
    o = hp.run_oracle(ps, blk, binding.ROWS_VARYING)
    S = blk.n_samples
    rows = {}
    for j in range(len(o["region"])):
        ir = blk.inner[int(o["inner"][j])]
        rid = "regions%d.bed,%s,%d-%d" % (int(ir["bed_index"]) + 1, name[int(o["pattern_id"][j])], int(ir["start"]), int(ir["end"]))
        rows[rid] = (int(o["region"][j]), int(o["inner"][j]) - int(blk.inner_off[o["region"][j]]), int(o["pattern_id"][j]),
                     int(o["left"][j].astype(np.int64).sum() + o["right"][j].astype(np.int64).sum()))
    assert set(ids) == set(rows)
    # sum over the lines of DIFF x HAPLOTYPES + 2 S x REF_COUNT = the oracle's sum of left + right
    total = {}
    for x in att:
        total[x["id"]] = total.get(x["id"], 2 * S * x["ref"]) + x["diff"] * x["haps"]
    for rid in ids:
        assert total[rid] == rows[rid][3], rid
    # DIFF and REF_COUNT of every line: the oracle on the region's window patched with the line's records alone
    by_region = {}
    for x in att:
        r = rows[x["id"]][0]
        v0, v1 = int(blk.var_off[r]), int(blk.var_off[r + 1])
        key = [(int(blk.variants["pos"][v]), bytes(blk.allele_bases[blk.variants["ref_off"][v]:blk.variants["ref_off"][v] + blk.variants["ref_len"][v]]).decode(),
                bytes(blk.allele_bases[blk.variants["alt_off"][v]:blk.variants["alt_off"][v] + blk.variants["alt_len"][v]]).decode()) for v in range(v0, v1)]
        recs = [v0 + key.index(rec) for rec in x["records"]]
        by_region.setdefault(r, []).append((x, recs))
    for r, items in by_region.items():
        configs = sorted(set(tuple(c) for _, c in items))
        diffs, ref = oracle_config_diffs(ps, blk, r, [list(c) for c in configs])
        for x, recs in items:
            k = rows[x["id"]][1:3]
            assert x["diff"] == diffs[configs.index(tuple(recs))].get(k, 0) != 0
            assert x["ref"] == ref.get(k, 0)
    # --audit and --attribution together are refused
    p = run_driver(files, str(tmp_path / "x.vcf.gz"), ["--attribution", path, "--audit", str(tmp_path / "a.tsv")])
    assert p.returncode != 0 and "--attribution" in (p.stdout + p.stderr)


@pytest.mark.gpu
def test_small_driver_reference_fixture(golden_dir, tmp_path):
    args = {"chromosome": "chr1", "bcf": os.path.join(golden_dir, "genotypes2.bcf"), "reference": os.path.join(golden_dir, "reference_genome.fa"),
            "beds": [os.path.join(golden_dir, "regions1.bed"), os.path.join(golden_dir, "regions2.bed")], "names": ["ACGT"],
            "pwm_file": os.path.join(golden_dir, "pwm_definitions.txt"), "threshold_dir": golden_dir,
            "extra": ["--samples", os.path.join(golden_dir, "samples")]}
    out, path = str(tmp_path / "out.vcf.gz"), str(tmp_path / "attribution.tsv")
    p = run_driver(args, out, ["--attribution", path])
    assert p.returncode == 0, p.stderr
    assert ora.gunzip_file(out) == ora.gunzip_file(os.path.join(golden_dir, "expected_output_2.vcf.gz"))  # the option changes no row
    att = read_attribution(path)
    check_driver_file(att, vcf_ids(out))
    # INDIVIDUAL1 = 1|0: its left haplotype carries the SNV at 100 (1-based 101), which destroys both ACGT hits of regions1.bed 100-110
    assert [(x["ref"], x["records"], x["diff"], x["haps"], x["trunc"]) for x in att] == [(2, [(100, "A", "G")], -2, 1, 0)]


# ---- large blocks (GPU only) --------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_configs2_shaped_block_on_a_few_regions():
    """A configs[2]-shaped block (2,504 samples, two BED sets, 401 PWMs) at 2 % of its regions: the block runs whole; the invariant
    and every term are checked on three of its regions against the oracle on those regions."""
    pats, blk = synth.config3(scale=0.02)
    ps = PatternSet(pats)
    g, a, st = run(ps, blk, binding.ROWS_VARYING)
    check_structure(with_block_arrays(g, blk), a)
    left, right = counts_from_attribution(g, a)
    counts = np.bincount(g["region"], minlength=blk.n_regions)
    picks = [int(r) for r in np.argsort(-counts, kind="stable")[:3]]
    for r in picks:
        sel = np.nonzero(g["region"] == r)[0]
        o = hp.run_oracle(ps, blk.slice(r, r + 1), binding.ROWS_VARYING, False, os.cpu_count() or 4)
        assert len(o["region"]) == len(sel) > 0
        assert np.array_equal(o["inner"] + blk.inner_off[r], g["inner"][sel]) and np.array_equal(o["pattern_id"], g["pattern_id"][sel])
        assert np.array_equal(left[sel], o["left"].astype(np.int64)) and np.array_equal(right[sel], o["right"].astype(np.int64))
    assert check_terms(ps, blk, g, a, regions=picks[:1]) > 0


@pytest.mark.gpu
def test_40000_samples_fanout_in_device_memory():
    """2 regions of 40,000 samples (about 80,000 groups each): the fan-out keeps its vectors in device memory."""
    pats = synth.make_pwms(4, seed=5, lmin=6, lmax=10, pvalue=1e-3)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(40000, 2, seed=5, lmax_pattern=lmax, region_len=(500, 700), variant_rate=1 / 4.0, gap=(100, 300))
    ps = PatternSet(pats)
    oracle = {mode: hp.run_oracle(ps, blk, mode, False, os.cpu_count() or 4, 1) for mode in MODES}
    check_invariant(ps, blk, oracle=oracle)
    ctx = binding.Context(0)
    try:
        ctx.set_option("attribution", 1)
        ctx.set_patterns(ps)
        ctx.submit_block(blk)
        ctx.collect_grouped()
        assert ctx.fanout_info()["in_device_memory"]
    finally:
        ctx.close()


# ---- the small cases on the emulated kernels (CPU) ----------------------------------------------------------------------------------

def test_small_cases_on_emulated_kernels():
    """The GPU tests named *small* on tests/cuda_emu/libtfbs_emu.so and the driver linked against it."""
    from test_large_regions import run_marked_gpu_tests
    subprocess.check_call(["make", "-C", EMU, "-j2", "libtfbs_emu.so", "find-tfbs-emu"], stdout=subprocess.DEVNULL)
    env = dict(os.environ, TFBS_B200_LIB=os.path.join(EMU, "libtfbs_emu.so"), TFBS_B200_DRIVER=os.path.join(EMU, "find-tfbs-emu"))
    out = run_marked_gpu_tests(env, "tests/test_attribution.py", "small")
    assert "14 passed" in out
