"""Per-group count vectors on both sides of the fan-out's shared-memory capacity, against a plain NumPy reference.

The fan-out builds one count per distinct haplotype (group) of a region.  A block whose count vector holds at most the groups that
fit in shared memory (tfbs_fanout_info: `smem_groups`) runs k_fanout<false>; a larger one keeps its count vectors in device memory
(k_fanout<true>).  Both must give the same counts, so the tests here compare every row of every region with `reference()`, a
restatement of the per-region computation written from the reference's rules (patch the window with a haplotype's records, score
every window of every pattern, count the windows whose hit range overlaps an inner region), not from the kernels' structure:

* sequences are patched like patch_haplotype (haplotype.rs:94-156): the ALT bases of an SNV or insertion all take the record's
  position, a deletion keeps its first ALT base and skips the rest of REF;
* a window of length L starting at sequence index i scores sum_c w[c][base(i + c)], N scoring 0, in float64; its hit range is
  (pos(i), pos(i) + L - 1) (pattern.rs:119-171);
* an inner region counts a hit when the hit's start or end lies inside it (range.rs:18-21, main.rs:500-534);
* haplotypes carrying the same records form one group; group 0 is the reference haplotype, the others are numbered in order of
  their smallest haplotype (the numbering tfbs_collect_grouped returns).

Threshold rule.  The project counts a window iff its score is STRICTLY above min_score (pattern.rs:151).  Weights and thresholds
are int32 and the kernels add them as exact integers, so there is no rounding anywhere: float64 holds every such sum exactly, the
reference computes the same score, and the comparison at ties is exact like everywhere else (no tolerance).  The tie tests put
window scores on the threshold, one unit and one float32 ulp of the threshold on either side, with scores large enough that a
float32 sum would not separate them.

Counts are compared with exact equality: the grouped rows (n_groups, the haplotype -> group map, every group's count) and the rows
expanded to samples, in both row modes, in the automatic fan-out and with the count vectors forced into device memory (option
fan_vector = 1).  The automatic run also asserts on which side of the capacity the fan-out ran.

The small cases run on the GPU and, through test_small_cases_on_emulated_kernels, on the kernels compiled for the host
(tests/cuda_emu); the cohorts at the capacity (up to 100,000 samples) run on the GPU only."""
import os

import numpy as np
import pytest

from find_tfbs_b200 import binding
from find_tfbs_b200.binding import INNER_DTYPE, VARIANT_DTYPE, Block, PatternSet

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODES = (binding.ROWS_VARYING, binding.ROWS_ALL_KEYS)
CODE = {c: i for i, c in enumerate("ACGTN")}
COMPLEMENT = np.array([3, 2, 1, 0])  # A<->T, C<->G


# ---- inputs ----------------------------------------------------------------------------------------------------------------------

class Region:
    """One window: reference bases (str) starting at `start`, inner regions [(first, last)] (inclusive), records [(pos, REF, ALT)]
    and carriers[v, h] = haplotype h carries record v."""

    def __init__(self, start, ref, inner, records=(), carriers=None, n_haps=0):
        self.start, self.ref, self.inner, self.records = start, ref, list(inner), list(records)
        self.carriers = np.zeros((len(self.records), n_haps), bool) if carriers is None else np.asarray(carriers, bool)
        self.codes = np.array([CODE[b] for b in ref.upper()], np.int64)
        assert self.carriers.shape[0] == len(self.records)


def make_block(regions, n_samples):
    H = 2 * n_samples
    pitch = max(1, (H + 31) // 32)
    starts = np.array([r.start for r in regions], np.int64)
    ends = np.array([r.start + len(r.ref) - 1 for r in regions], np.int64)
    ref_off = np.concatenate([[0], np.cumsum([len(r.ref) for r in regions])]).astype(np.uint64)
    ref_bases = np.frombuffer("".join(r.ref for r in regions).encode(), np.uint8)
    inner_off = np.concatenate([[0], np.cumsum([len(r.inner) for r in regions])]).astype(np.uint32)
    inner = np.zeros(int(inner_off[-1]), INNER_DTYPE)
    inner["start"] = [a for r in regions for a, _ in r.inner]
    inner["end"] = [b for r in regions for _, b in r.inner]
    inner["multiplicity"] = 1
    var_off = np.concatenate([[0], np.cumsum([len(r.records) for r in regions])]).astype(np.uint32)
    variants = np.zeros(int(var_off[-1]), VARIANT_DTYPE)
    alleles, rows = bytearray(), []
    for i, (pos, ref, alt) in enumerate(rec for r in regions for rec in r.records):
        variants[i] = (pos, len(alleles), len(ref), len(alleles) + len(ref), len(alt), i, 0)
        alleles += (ref + alt).encode()
    for r in regions:
        assert r.carriers.shape[1] == H
        if len(r.records):
            bits = np.zeros((len(r.records), pitch * 32), bool)
            bits[:, :H] = r.carriers
            rows.append(np.packbits(bits, axis=1, bitorder="little").view("<u4"))
    carriers = np.concatenate(rows) if rows else np.zeros((1, pitch), np.uint32)
    return Block(n_samples, starts, ends, ref_off, ref_bases, inner_off, inner, var_off, variants, np.frombuffer(bytes(alleles), np.uint8),
                 carriers)


def pwm(weights, min_score, pattern_id, both_strands=True):
    """A pattern, and its reverse complement under the same pattern_id (how the reference lists the two strands)."""
    w = np.asarray(weights, np.int32)
    pats = [{"weights": w, "min_score": int(min_score), "pattern_id": pattern_id}]
    if both_strands:
        pats.append({"weights": np.ascontiguousarray(w[::-1][:, COMPLEMENT]), "min_score": int(min_score), "pattern_id": pattern_id,
                     "direction": binding.DIR_N})
    return pats


def consensus_pwm(consensus, max_mismatches, pattern_id):
    """+30 for the consensus base, -10 otherwise: a window hits with at most `max_mismatches` mismatches."""
    w = np.full((len(consensus), 4), -10, np.int32)
    for c, b in enumerate(consensus):
        w[c, CODE[b]] = 30
    return pwm(w, 30 * len(consensus) - 40 * max_mismatches - 1, pattern_id)


# ---- the reference ------------------------------------------------------------------------------------------------------------------

def patch(region, carried):
    """Bases (codes 0..4) and positions of the window patched with the records `carried` (non-overlapping, inside the window)."""
    codes = region.codes
    end = region.start + len(region.ref) - 1
    seq, pos, p = [], [], region.start
    for v in sorted(carried, key=lambda v: region.records[v]):
        vpos, ref, alt = region.records[v]
        assert p <= vpos <= end, "overlapping records are out of the reference's scope"
        assert codes[vpos - region.start] == CODE[ref[0]]
        seq.append(codes[p - region.start:vpos - region.start])
        pos.append(np.arange(p, vpos))
        if len(ref) == 1:  # SNV or insertion: every ALT base at the record's position
            seq.append(np.array([CODE[b] for b in alt]))
            pos.append(np.full(len(alt), vpos))
            p = vpos + 1
        else:  # deletion
            assert len(alt) == 1
            seq.append(np.array([CODE[alt]]))
            pos.append(np.array([vpos]))
            p = vpos + len(ref)
    if p <= end:
        seq.append(codes[p - region.start:])
        pos.append(np.arange(p, end + 1))
    return np.concatenate(seq).astype(np.int64), np.concatenate(pos).astype(np.int64)


def window_scores(seqs, weights):
    """float64 scores of every window of every row of seqs (n, len): (n, len - L + 1); N scores 0."""
    w = np.zeros((len(weights), 5))
    w[:, :4] = weights
    L, n = len(weights), seqs.shape[1] - len(weights) + 1
    out = np.zeros((seqs.shape[0], max(0, n)))
    for c in range(L if n > 0 else 0):
        out += w[c][seqs[:, c:c + n]]
    return out


def group_haplotypes(carriers):
    """Group of every haplotype: 0 = carries nothing, then distinct record sets in order of their smallest haplotype."""
    V, H = carriers.shape
    if V == 0:
        return np.zeros(H, np.int64), []
    keys = np.packbits(carriers.T, axis=1)
    uniq, first, inv = np.unique(keys, axis=0, return_index=True, return_inverse=True)
    inv = inv.reshape(-1)
    carried = [np.nonzero(np.unpackbits(u)[:V])[0] for u in uniq]
    order = [u for u in np.argsort(first, kind="stable") if len(carried[u])]
    number = np.zeros(len(uniq), np.int64)
    number[order] = np.arange(1, len(order) + 1)
    return number[inv], [carried[u] for u in order]


def region_counts(region, patterns, pids, ge=False):
    """(hap_group, counts[group, key]) of one region; key = pid index * n_inner + inner index.  ge=True counts score >= min_score
    instead of the project's strict rule (used only to show that a test separates the two)."""
    hap_group, sets = group_haplotypes(region.carriers)
    n_inner = len(region.inner)
    counts = np.zeros((len(sets) + 1, len(pids) * n_inner), np.int64)
    if all(len(r) == 1 and len(a) == 1 for _, r, a in region.records):  # SNVs only: every sequence has the window's positions
        S = np.tile(region.codes, (len(sets) + 1, 1))
        for g, carried in enumerate(sets, 1):
            for v in carried:
                pos, _, alt = region.records[v]
                S[g, pos - region.start] = CODE[alt]
        batches = [(list(range(len(sets) + 1)), S, np.tile(np.arange(region.start, region.start + len(region.ref)), (len(sets) + 1, 1)))]
        assert len(np.unique(S, axis=0)) == len(S)
    else:
        seqs = [patch(region, [])] + [patch(region, s) for s in sets]
        assert len({(s.tobytes(), p.tobytes()) for s, p in seqs}) == len(seqs), "two record sets patch to one sequence: out of scope"
        by_len = {}
        for g, (s, p) in enumerate(seqs):
            by_len.setdefault(len(s), []).append(g)
        batches = [(gs, np.stack([seqs[g][0] for g in gs]), np.stack([seqs[g][1] for g in gs])) for gs in by_len.values()]
    for gs, S, P in batches:
        for pat in patterns:
            sc = window_scores(S, pat["weights"])
            if sc.shape[1] == 0:
                continue
            hit = sc >= pat["min_score"] if ge else sc > pat["min_score"]
            first = P[:, :sc.shape[1]]
            last = first + len(pat["weights"]) - 1
            k0 = pids.index(pat["pattern_id"]) * n_inner
            a = np.array([x for x, _ in region.inner])
            b = np.array([y for _, y in region.inner])
            if (P == P[0]).all():  # one set of hit ranges for the whole batch: count by a product with the overlap matrix
                f, l = first[0][:, None], last[0][:, None]
                over = ((f >= a) & (f <= b)) | ((l >= a) & (l <= b))
                counts[gs, k0:k0 + n_inner] += hit.astype(np.int64) @ over.astype(np.int64)
                continue
            for i in range(n_inner):
                over = ((first >= a[i]) & (first <= b[i])) | ((last >= a[i]) & (last <= b[i]))
                counts[gs, k0 + i] += (hit & over).sum(axis=1)
    return hap_group, counts


def reference(regions, patterns, ge=False):
    pids = sorted({p["pattern_id"] for p in patterns})
    out = []
    for r in regions:
        hg, counts = region_counts(r, patterns, pids, ge)
        out.append({"hap_group": hg, "counts": counts, "n_groups": counts.shape[0], "pids": pids})
    return out


def expected_rows(regions, ref, mode):
    rows = {k: [] for k in ("region", "inner", "pattern_id", "vmin", "vmax", "left", "right", "group_counts")}
    inner0 = 0
    for r, (reg, e) in enumerate(zip(regions, ref)):
        n_inner = len(reg.inner)
        per_hap = e["counts"][e["hap_group"]]  # (H, keys)
        for k in range(per_hap.shape[1]):
            c = per_hap[:, k]
            v = c[0::2] + c[1::2]
            keep = (c.max() > 0) if mode == binding.ROWS_ALL_KEYS else (v.min() != v.max())
            if not keep:
                continue
            rows["region"].append(r)
            rows["inner"].append(inner0 + k % n_inner)
            rows["pattern_id"].append(e["pids"][k // n_inner])
            rows["vmin"].append(v.min())
            rows["vmax"].append(v.max())
            rows["left"].append(c[0::2])
            rows["right"].append(c[1::2])
            rows["group_counts"].append(e["counts"][:, k])
        inner0 += n_inner
    return rows


# ---- running and comparing ----------------------------------------------------------------------------------------------------------

def group_counts(g, j):
    """Count of every group of row j of grouped rows."""
    n = int(g["n_groups"][g["region"][j]])
    bits, base = int(g["bits"][j]), int(g["base"][j])
    if bits == 0:
        return np.full(n, base, np.int64)
    at = np.arange(n, dtype=np.int64) * bits
    words = g["packed"][int(g["offset"][j]) + (at >> 5)].astype(np.int64)
    return base + ((words >> (at & 31)) & ((1 << bits) - 1))


def run(regions, n_samples, patterns, mode, fan_vector=0, options=None):
    blk = make_block(regions, n_samples)
    ctx = binding.Context(0)
    try:
        ctx.set_option("rows_mode", mode)
        ctx.set_option("fan_vector", fan_vector)
        for k, v in (options or {}).items():
            ctx.set_option(k, v)
        ctx.set_patterns(PatternSet(patterns))
        ctx.submit_block(blk)
        g = binding.own_grouped(ctx.collect_grouped(expand=True))
        g["fan"] = ctx.fanout_info()
        return g
    finally:
        ctx.close()


def compare(regions, n_samples, patterns, ref=None, modes=MODES, fan_vectors=(0, 1), options=None):
    """Every mode x fan-out variant equals the reference exactly; returns the fan-out info of every run."""
    ref = reference(regions, patterns) if ref is None else ref
    fans = []
    for mode in modes:
        exp = expected_rows(regions, ref, mode)
        for fv in fan_vectors:
            g = run(regions, n_samples, patterns, mode, fv, options)
            where = "mode %d fan_vector %d" % (mode, fv)
            assert [int(x) for x in g["n_groups"]] == [e["n_groups"] for e in ref], where
            for r, e in enumerate(ref):
                assert np.array_equal(np.asarray(g["hap_group"][r], np.int64), e["hap_group"]), "%s: haplotype -> group map of region %d" % (where, r)
            assert len(g["region"]) == len(exp["region"]), "%s: %d rows, expected %d" % (where, len(g["region"]), len(exp["region"]))
            for k in ("region", "inner", "pattern_id", "vmin", "vmax"):
                assert np.array_equal(np.asarray(g[k], np.int64), np.asarray(exp[k], np.int64)), "%s: rows differ in %s" % (where, k)
            for j in range(len(exp["region"])):
                r = exp["region"][j]
                assert np.array_equal(group_counts(g, j), exp["group_counts"][j]), "%s: group counts of row %d (region %d)" % (where, j, r)
                assert np.array_equal(g["left"][j], exp["left"][j]) and np.array_equal(g["right"][j], exp["right"][j]), \
                    "%s: sample counts of row %d (region %d)" % (where, j, r)
            if fv:
                assert g["fan"]["in_device_memory"]
            fans.append(dict(g["fan"], forced=bool(fv)))
    return fans


def assert_side(fans, max_groups):
    """The automatic fan-out ran in shared memory iff the block's largest region fits a shared-memory count vector."""
    for f in fans:
        if f["forced"]:
            continue
        assert f["groups_cap"] >= max_groups
        assert f["in_device_memory"] == (max_groups > f["smem_groups"]), (f, max_groups)
        if not f["in_device_memory"]:
            assert f["groups_cap"] <= f["smem_groups"]


def random_bases(rng, n, alphabet="ACGT"):
    return "".join(rng.choice(list(alphabet), n))


def snv_records(rng, region_start, ref, positions):
    recs = []
    for p in positions:
        b = ref[p]
        recs.append((region_start + p, b, rng.choice([x for x in "ACGT" if x != b])))
    return recs


# ---- cohorts at the shared-memory capacity (GPU) ------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def smem_groups():
    ctx = binding.Context(0)
    try:
        return ctx.fanout_info()["smem_groups"]
    finally:
        ctx.close()


CAPACITY_MOTIFS = consensus_pwm("ACGTTGCA", 4, 1) + consensus_pwm("TTAGGC", 2, 2)


def capacity_region(n_groups, n_haps, seed, start, n_inner=2):
    """A 64-bp window with 18 SNVs (2^18 - 1 record sets) whose haplotypes form exactly n_groups groups (the reference haplotype
    included): n_groups - 1 distinct record sets, the other haplotypes carry nothing or repeat one of them.  Two inner regions, or
    n_inner overlapping ones."""
    rng = np.random.default_rng(seed)
    ref = random_bases(rng, 64)
    recs = snv_records(rng, start, ref, sorted(rng.choice(np.arange(1, 63), 18, replace=False)))
    assert n_groups - 1 <= n_haps
    codes = rng.choice(np.arange(1, 1 << 18), n_groups - 1, replace=False)
    hap = np.zeros(n_haps, np.int64)
    perm = rng.permutation(n_haps)
    hap[perm[:n_groups - 1]] = codes
    if n_groups > 1:
        rest = perm[n_groups - 1:]
        hap[rest[::2]] = rng.choice(codes, len(rest[::2]))
    carriers = ((hap[None, :] >> np.arange(18)[:, None]) & 1).astype(bool)
    inner = [(start + 5, start + 30), (start + 28, start + 60)] if n_inner == 2 else [(start + 3 * i, start + 3 * i + 12) for i in range(n_inner)]
    return Region(start, ref, inner, recs, carriers)


def check_last_group_differs(ref):
    """The test data touches the vector's last entry: in every region of 1,000 groups or more, the highest group's counts differ from
    the reference haplotype's."""
    for e in ref:
        if e["n_groups"] >= 1000:
            assert (e["counts"][-1] != e["counts"][0]).any()


CAPACITY_POINTS = {"1": lambda c: 1, "cap-1": lambda c: c - 1, "cap": lambda c: c, "cap+1": lambda c: c + 1, "2cap": lambda c: 2 * c,
                   "2cap+1": lambda c: 2 * c + 1}


@pytest.mark.gpu
@pytest.mark.parametrize("point", list(CAPACITY_POINTS))
def test_capacity_boundary(point, smem_groups):
    """One region with 1, capacity - 1, capacity, capacity + 1, 2 x capacity and 2 x capacity + 1 groups: shared memory up to the
    capacity, device memory above it, both equal to the reference."""
    n = CAPACITY_POINTS[point](smem_groups)
    S = n // 2 + 40
    regions = [capacity_region(n, 2 * S, seed=100 + n, start=5000)]
    ref = reference(regions, CAPACITY_MOTIFS)
    assert ref[0]["n_groups"] == n
    check_last_group_differs(ref)
    assert_side(compare(regions, S, CAPACITY_MOTIFS, ref), n)


@pytest.mark.gpu
def test_cohort_size_region():
    """100,000 samples, every haplotype distinct: 200,001 groups in one region, nearly four times the capacity."""
    S = 100000
    regions = [capacity_region(2 * S + 1, 2 * S, seed=7, start=9000)]
    ref = reference(regions, CAPACITY_MOTIFS)
    assert ref[0]["n_groups"] == 200001
    check_last_group_differs(ref)
    assert_side(compare(regions, S, CAPACITY_MOTIFS, ref, modes=(binding.ROWS_ALL_KEYS,)), 200001)


def assert_slices_reused(fans, n_regions):
    """The device-memory fan-out ran with fewer CTAs than the block has regions.  Every region has keys, so its first unit has work,
    and the CTAs walk the units in a grid-stride loop: some CTA ran units of two regions in its one count vector."""
    for f in fans:
        assert f["in_device_memory"] and 0 < f["ctas"] < n_regions, (f, n_regions)


@pytest.mark.gpu
def test_large_regions_in_one_launch(smem_groups):
    """Three regions above the capacity, of different sizes, first, in the middle and last, between 297 small regions: one launch of
    the device-memory fan-out with more regions than CTAs, so CTAs run several regions in their count vector one after the other.
    Every region equals its own reference: counts left behind in a vector, or written to another CTA's, would show."""
    c = smem_groups
    sizes = [c + c // 2] + [2 + i % 60 for i in range(148)] + [c + 1] + [2 + i % 45 for i in range(149)] + [2 * c + 1]
    S = c + 80
    regions = [capacity_region(n, 2 * S, seed=300 + i, start=20000 + 1000 * i) for i, n in enumerate(sizes)]
    ref = reference(regions, CAPACITY_MOTIFS)
    assert [e["n_groups"] for e in ref] == sizes
    check_last_group_differs(ref)
    fans = compare(regions, S, CAPACITY_MOTIFS, ref, fan_vectors=(0,))
    assert_side(fans, max(sizes))
    assert_slices_reused(fans, len(regions))


@pytest.mark.gpu
def test_slices_filled_and_reused():
    """320 regions of exactly 2,048 groups and 32 keys each, count vectors forced into device memory: a cold context gives the vector
    2,048 groups, so every region fills its CTA's slice to the last word (the slice is 2,048 words wide), and the regions outnumber
    the CTAs, so every slice is reused.  A slice offset or stride one word off makes neighbouring CTAs' vectors overlap."""
    S, n, R = 1100, 2048, 320
    regions = [capacity_region(n, 2 * S, seed=900 + i, start=50000 + 1000 * i, n_inner=16) for i in range(R)]
    ref = reference(regions, CAPACITY_MOTIFS)
    assert all(e["n_groups"] == n for e in ref)
    check_last_group_differs(ref)
    fans = compare(regions, S, CAPACITY_MOTIFS, ref, fan_vectors=(1,))
    assert all(f["groups_cap"] == n for f in fans)
    assert_slices_reused(fans, R)


# ---- small cases (GPU; also on the emulated kernels) -----------------------------------------------------------------------------

def random_carriers(rng, V, H, p):
    return rng.random((V, H)) < p


@pytest.mark.gpu
def test_small_mixed_regions_in_one_launch():
    """Small and larger regions mixed in one block (large first, in the middle and last), with the count vectors in device memory
    (forced) and in shared memory.  (On the emulated device, 3 SMs, the 7 regions outnumber the fan-out's CTAs; on a B200 they do
    not: test_large_regions_in_one_launch and test_slices_filled_and_reused reuse the device-memory vectors there.)"""
    rng = np.random.default_rng(11)
    S = 150
    regions = []
    for i, big in enumerate([True, False, False, True, False, True, False]):
        ref = random_bases(rng, 300 if big else 50)
        V = 14 if big else 2
        recs = snv_records(rng, 1000 * (i + 1), ref, sorted(rng.choice(np.arange(len(ref)), V, replace=False)))
        regions.append(Region(1000 * (i + 1), ref, [(1000 * (i + 1) + 10, 1000 * (i + 1) + len(ref) - 20)], recs,
                              random_carriers(rng, V, 2 * S, 0.3 if big else 0.2)))
    pats = consensus_pwm("ACGTTGCA", 4, 1) + consensus_pwm("TTAGGC", 2, 2)
    ref = reference(regions, pats)
    assert min(e["n_groups"] for e in ref) < 5 and max(e["n_groups"] for e in ref) > 200
    assert_side(compare(regions, S, pats, ref), max(e["n_groups"] for e in ref))


EDGE_MOTIF = consensus_pwm("ACGTTG", 1, 1)


def edge_case(name):
    """(regions, n_samples) of one data edge; 6 samples = 12 haplotypes."""
    S, H = 6, 12
    rng = np.random.default_rng(EDGES.index(name))
    alt = np.zeros((1, H), bool)
    alt[0, [1, 4, 5, 10]] = True
    if name == "shorter_than_motif":
        return [Region(100, "ACGT", [(100, 103)], [(101, "C", "A")], alt)], S
    if name == "one_motif_long":  # the consensus: one window, a hit; two SNVs break it on their carriers
        return [Region(100, "ACGTTG", [(100, 105)], [(102, "G", "T"), (103, "T", "A")], np.concatenate([alt, alt]))], S
    if name == "first_and_last_base":  # SNVs on the first and the last base, an insertion at the last base
        ref = "ACGTTG" + random_bases(rng, 28) + "CAACGT"
        c = np.zeros((3, H), bool)
        c[0, [0, 3, 7]] = c[1, [3, 8]] = c[2, [2, 9, 11]] = True
        end = 100 + len(ref) - 1
        return [Region(100, ref, [(100, 110), (end - 8, end)], [(100, "A", "T"), (end, "T", "C"), (end, "T", "TTG")], c)], S
    if name == "indel_across_boundary":
        # inner region [110, 125].  A deletion joins ACG|TTG across two junk bases: the new site starts at 123, inside.  An insertion
        # at 125 puts a whole site at position 125 = the inner region's last base.  A deletion near the window's end runs past it.
        ref = "GGGGGGGGGG" + "CCCCCCCCCCCCC" + "ACG" + "CC" + "TTG" + "GGGGGGGGGG" + "CCCCC"
        end = 100 + len(ref) - 1
        c = np.zeros((3, H), bool)
        c[0, [0, 2, 5, 6]] = c[1, [1, 5, 7, 11]] = c[2, [3, 6, 9]] = True
        c[1, 5] = False  # the deletion and the insertion share a position: no haplotype carries both
        return [Region(100, ref, [(110, 125)], [(125, "GCC", "G"), (125, "G", "GACGTTG"), (end - 1, "CCCC", "C")], c)], S
    if name == "all_identical":  # every haplotype carries the same two records: one distinct haplotype
        ref = random_bases(rng, 10) + "ACGTTG" + random_bases(rng, 24)
        return [Region(100, ref, [(105, 130)], snv_records(rng, 100, ref, [12, 30]), np.ones((2, H), bool))], S
    if name == "all_distinct":  # 12 haplotypes, 12 different record sets of 4 records
        ref = "ACGTTGAC" + random_bases(rng, 30) + "CAACGT"
        recs = snv_records(rng, 100, ref, [2, 5, 20, 40])
        codes = np.arange(1, H + 1)
        return [Region(100, ref, [(100, 143)], recs, ((codes[None, :] >> np.arange(4)[:, None]) & 1).astype(bool))], S
    if name == "no_sites":  # no window of any haplotype reaches the threshold
        ref = "TTTTTTTTTTTTTTTTTTTTTTTTT"
        return [Region(100, ref, [(100, 124)], [(110, "T", "G"), (115, "T", "C")], random_carriers(rng, 2, H, 0.5))], S
    raise KeyError(name)


EDGES = ["shorter_than_motif", "one_motif_long", "first_and_last_base", "indel_across_boundary", "all_identical", "all_distinct",
         "no_sites"]


def test_edge_cases_are_what_they_claim():
    """The reference on the edge data (CPU): each case has the property its name states."""
    def ref_of(name):
        regions, _ = edge_case(name)
        return regions, reference(regions, EDGE_MOTIF)
    regions, e = ref_of("shorter_than_motif")
    assert len(regions[0].ref) < 6 and not e[0]["counts"].any()
    regions, e = ref_of("one_motif_long")
    assert e[0]["counts"][0].tolist() == [1] and e[0]["counts"][1].tolist() == [0]
    regions, e = ref_of("indel_across_boundary")
    assert e[0]["counts"][0, 0] < e[0]["counts"][1:, 0].max()  # the indels create sites the inner region counts
    regions, e = ref_of("all_identical")
    assert e[0]["n_groups"] == 2 and (e[0]["hap_group"] == 1).all() and e[0]["counts"][1].any()
    regions, e = ref_of("all_distinct")
    assert e[0]["n_groups"] == 13 and sorted(e[0]["hap_group"]) == list(range(1, 13))
    regions, e = ref_of("no_sites")
    assert not e[0]["counts"].any()


@pytest.mark.gpu
@pytest.mark.parametrize("name", EDGES)
def test_small_data_edge(name):
    regions, S = edge_case(name)
    compare(regions, S, EDGE_MOTIF)


@pytest.mark.gpu
def test_small_data_edges_in_one_block():
    regions, S = [], 6
    for i, name in enumerate(EDGES):
        for r in edge_case(name)[0]:
            shift = 1000 * (i + 1)
            regions.append(Region(r.start + shift, r.ref, [(a + shift, b + shift) for a, b in r.inner],
                                  [(p + shift, x, y) for p, x, y in r.records], r.carriers))
    compare(regions, S, EDGE_MOTIF)


# ---- threshold ties ------------------------------------------------------------------------------------------------------------------

def tie_patterns(K):
    """Length 4, base deficits 0 / 1 / 4 / 8 per column below K: a window scores 4K - (sum of deficits).  min_score = 4K - 4."""
    w = np.array([[K, K - 1, K - 4, K - 8]] * 4, np.int64)
    return [{"weights": w.astype(np.int32), "min_score": int(4 * K - 4), "pattern_id": 3}]


def tie_regions(S):
    rng = np.random.default_rng(21)
    regions = []
    for i in range(2):
        ref = random_bases(rng, 600)
        recs = snv_records(rng, 500 + 1000 * i, ref, sorted(rng.choice(np.arange(600), 40, replace=False)))
        regions.append(Region(500 + 1000 * i, ref, [(500 + 1000 * i, 1099 + 1000 * i), (700 + 1000 * i, 720 + 1000 * i)], recs,
                              random_carriers(rng, 40, 2 * S, 0.15)))
    return regions


@pytest.mark.parametrize("K", [100, (1 << 23) + (1 << 21)])
def test_tie_data_lands_on_the_threshold(K):
    """CPU: the tie data has windows at min_score, at +-1 and at +-one float32 ulp of it (K = 2^23 + 2^21: scores near 2^25, where a
    float32 ulp is 4 and a float32 sum could not tell min_score from min_score + 1); counting >= instead of > changes the rows."""
    pats = tie_patterns(K)
    T = pats[0]["min_score"]
    regions = tie_regions(8)
    seqs = [patch(r, s) for r in regions for s in [[]] + group_haplotypes(r.carriers)[1]]
    scores = np.concatenate([window_scores(s[None, :], pats[0]["weights"])[0] for s, _ in seqs])
    ulp = float(np.spacing(np.float32(T)))
    steps = (1, ulp) if ulp >= 1 else (1,)
    for d in (0,) + tuple(x for st in steps for x in (-st, st)):
        assert (scores == T + d).any(), d
    if K > 1000:
        assert ulp == 4 and np.float32(T) == np.float32(T + 1)
    strict, ge = reference(regions, pats), reference(regions, pats, ge=True)
    assert any((a["counts"] != b["counts"]).any() for a, b in zip(strict, ge))


@pytest.mark.gpu
@pytest.mark.parametrize("K", [100, (1 << 23) + (1 << 21)])
def test_small_threshold_ties(K):
    """Exact equality at the ties: 21-bit table fields (K = 100) and 32-bit fields (scores near 2^25)."""
    compare(tie_regions(8), 8, tie_patterns(K))


# ---- high counts --------------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_small_high_counts():
    """One motif that hits almost every window of both strands (no A or T in the window) of 1,500-bp windows, 400 samples with many
    records apart from each other: thousands of hits per haplotype, each configuration's differences added into the groups with
    atomics.  A lost or repeated increment changes a count."""
    rng = np.random.default_rng(5)
    S = 400
    w = np.array([[-50, 5, 5, -50]] * 6, np.int32)
    pats = pwm(w, 0, 9)
    regions = []
    for i in range(2):
        n = 1500
        ref = "".join(rng.choice(list("CG"), n))
        ref = "".join(b if rng.random() > 0.01 else rng.choice(list("AT")) for b in ref)
        positions = np.arange(20, n - 20, 37)
        recs = []
        for p in positions:
            b = ref[p]
            recs.append((10000 * (i + 1) + int(p), b, rng.choice(list("AT")) if b in "CG" else rng.choice(list("CG"))))
        start = 10000 * (i + 1)
        regions.append(Region(start, ref, [(start, start + n - 1), (start + 400, start + 460)], recs,
                              random_carriers(rng, len(recs), 2 * S, 0.25)))
    ref = reference(regions, pats)
    assert min(int(e["counts"][:, 0].min()) for e in ref) > 2000
    assert max(e["n_groups"] for e in ref) > 700
    compare(regions, S, pats, ref)


# ---- the small cases on the emulated kernels (CPU) --------------------------------------------------------------------------------

def test_small_cases_on_emulated_kernels():
    """The GPU tests named *small* on tests/cuda_emu/libtfbs_emu.so (the product's kernel sources on a CUDA-on-host shim)."""
    import subprocess
    from test_large_regions import EMU, run_marked_gpu_tests
    subprocess.check_call(["make", "-C", EMU, "-j2", "libtfbs_emu.so"], stdout=subprocess.DEVNULL)
    env = dict(os.environ, TFBS_B200_LIB=os.path.join(EMU, "libtfbs_emu.so"))
    out = run_marked_gpu_tests(env, "tests/test_haplotype_capacity.py", "small")
    assert "%d passed" % (len(EDGES) + 5) in out
