"""The PWM scan at the edges of its packed tables and of its window staging, against the plain NumPy reference of
test_haplotype_capacity.py.

k_scan adds up packed table words (three 21-bit or two 32-bit biased fields per word, tables.cpp) and decides a hit from one bit
per field; the rare path then keeps complete windows only, and the configuration path scores a patched haplotype only at the window
starts that touch one of its records.  Every one of these steps has an off-by-one that random data reaches only by chance, so each
case here is built to sit exactly on one edge:

* fields: a 21-bit field exactly full (bmax - thr = 2^20; thr = 2^20 - 1), one past it (the list switches to 32-bit fields), a
  32-bit field exactly full (bmax - thr = 2^31), with the next slot of the word scoring exactly its min_score on the window that
  fills the field, so that a carry out of the field shows up as a false hit;
* thresholds at M - 1, M, M + bmax - 1 and M + bmax (always-hit, tie at the worst window, only the best window, never-hit), where M
  is the sum of the column minima (N included, it scores 0);
* columns whose four weights share one sign, so that N is the column's unique best or worst base, in both halves of a column pair;
* every run length G = 1..16 and every slot count, chunks of one or two pattern ids, sequence, piece and tile ends;
* the configuration path's windows next to an ALT segment, a deletion junction and a cluster cut, a configuration item of more
  than 1,024 starts whose staging starts at p0 % 32 == 31, more configurations than one warp round takes;
* inner regions strictly inside a hit (not counted, range.rs:18-21) next to ones touching its first or last base (counted), with
  multiplicity 3, on a reference hit that a configuration loses and on a hit that a configuration gains.

Every case runs through the C ABI in both scan modes and must match exactly: the full scan (record_matches) against the reference's
hit list and hit count, the default configuration path against the reference's rows (both row modes).
test_scan_edges_are_what_they_claim checks on the CPU that each case really reaches its edge.  The *small* tests also run on the
emulated kernels (test_scan_edges_on_emulated_kernels)."""
import os

import numpy as np
import pytest

from find_tfbs_b200 import binding
from find_tfbs_b200.binding import PatternSet
from test_haplotype_capacity import (CODE, MODES, Region, compare, expected_rows, group_haplotypes, make_block, patch, reference,
                                     window_scores)

H21, H32 = 1 << 20, 1 << 31
PAIR_WORDS = 25


# ---- the reference's hit list ----------------------------------------------------------------------------------------------------

def scanned(region):
    """(group, bases, positions) of every distinct haplotype of the region, group 0 = the reference haplotype."""
    _, sets = group_haplotypes(region.carriers)
    return [(g, *patch(region, s)) for g, s in enumerate([[]] + sets)]


def reference_hits(regions, patterns, tie=False):
    """Sorted (region, pattern index, group, start) of every complete window scoring above min_score (tie=True: exactly
    min_score) in every distinct haplotype, groups numbered like tfbs_get_matches.  The reference haplotype is scanned only when a
    haplotype carries none of the region's records."""
    out = []
    for r, reg in enumerate(regions):
        present = set(group_haplotypes(reg.carriers)[0].tolist())
        for g, seq, pos in scanned(reg):
            if g not in present:
                continue
            for pi, p in enumerate(patterns):
                if p.get("kind", binding.PATTERN_PWM) != binding.PATTERN_PWM:
                    continue
                sc = window_scores(seq[None, :], p["weights"])[0]
                sel = sc == p["min_score"] if tie else sc > p["min_score"]
                out += [(r, pi, g, int(pos[i])) for i in np.nonzero(sel)[0]]
    return sorted(out)


def table_rows(m):
    return sorted(zip(*(np.asarray(m[k], np.int64).tolist() for k in ("region", "pattern_index", "group", "start"))))


def run_full(regions, n_samples, patterns, options=None):
    blk = make_block(regions, n_samples)
    ctx = binding.Context(0)
    try:
        ctx.set_option("rows_mode", binding.ROWS_ALL_KEYS)
        ctx.set_option("record_matches", 1)
        for k, v in (options or {}).items():
            ctx.set_option(k, v)
        ctx.set_patterns(PatternSet(patterns))
        ctx.submit_block(blk)
        rows = ctx.collect()
        return rows, ctx.matches(len(regions)), ctx.stats()
    finally:
        ctx.close()


def check(regions, n_samples, patterns, options=None, launches=None):
    """Full scan: hit list, hit count and rows; default path: grouped and expanded rows in both row modes."""
    ref = reference(regions, patterns)
    hits = reference_hits(regions, patterns)
    rows, m, st = run_full(regions, n_samples, patterns, options)
    assert not m["truncated"]
    hg = m["hap_group"].reshape(len(regions), -1)
    for r, e in enumerate(ref):
        assert np.array_equal(hg[r].astype(np.int64), e["hap_group"]), "full scan: haplotype -> group map of region %d" % r
    got = table_rows(m)
    if got != hits:
        extra, lost = sorted(set(got) - set(hits)), sorted(set(hits) - set(got))
        raise AssertionError("full scan: %d hits, expected %d; not expected %s; missing %s" % (len(got), len(hits), extra[:8], lost[:8]))
    assert st["n_hits"] == len(hits)
    if launches is not None:
        assert st["scan_launches"] == launches
    exp = expected_rows(regions, ref, binding.ROWS_ALL_KEYS)
    assert len(rows["region"]) == len(exp["region"])
    for k in ("region", "inner", "pattern_id", "vmin", "vmax", "left", "right"):
        assert np.array_equal(np.asarray(rows[k], np.int64), np.asarray(exp[k], np.int64)), "full scan: rows differ in " + k
    compare(regions, n_samples, patterns, ref, fan_vectors=(0,), options=options)
    return hits


# ---- building blocks ------------------------------------------------------------------------------------------------------------

def pat(weights, min_score, pid, direction=binding.DIR_P):
    return {"weights": np.asarray(weights, np.int32), "min_score": int(min_score), "pattern_id": pid, "direction": direction}


def revcomp_pat(p):
    return dict(p, weights=np.ascontiguousarray(p["weights"][::-1][:, [3, 2, 1, 0]]), direction=binding.DIR_N)


def plan(p):
    """(M, bmax) of tables.cpp's plan_field: column minima and maxima with the N slot (0) included."""
    w = np.asarray(p["weights"], np.int64)
    lo, hi = np.minimum(w.min(axis=1), 0), np.maximum(w.max(axis=1), 0)
    return int(lo.sum()), int((hi - lo).sum())


def fits(p, bits):
    M, bmax = plan(p)
    thr = p["min_score"] - M
    return thr < 0 or thr >= bmax or (thr <= (1 << (bits - 1)) - 1 and bmax - thr <= 1 << (bits - 1))


def bases(codes):
    return "".join("ACGTN"[c] for c in codes)


def random_bases(rng, n, alphabet="ACGT", n_rate=0.0):
    s = rng.choice(list(alphabet), n)
    if n_rate:
        s[rng.random(n) < n_rate] = "N"
    return "".join(s)


def put(ref, at, s):
    return ref[:at] + s + ref[at + len(s):]


def quantile_threshold(regions, p, q):
    sc = np.concatenate([window_scores(seq[None, :], p["weights"])[0] for r in regions for _, seq, _ in scanned(r)])
    return int(np.quantile(sc, q)) if len(sc) else 0


def consensus(s, mismatches=0, pid=1, direction=binding.DIR_P):
    """+10 for the consensus base, -10 otherwise: a window hits with at most `mismatches` mismatches."""
    w = np.full((len(s), 4), -10, np.int32)
    for c, b in enumerate(s):
        w[c, CODE[b]] = 10
    return pat(w, 10 * len(s) - 20 * mismatches - 1, pid, direction)


# ---- field capacity: slot 0 fills its field on a planted window, slot 1 ties there ------------------------------------------------

BEST, WORST, THIRD = [0, 1, 2, 3], [3, 2, 0, 1], [2, 3, 1, 0]
FIELD_SETS = {  # (bits of the field slot 0 is built for, thr = min_score - M)
    "full21": (21, H21 // 2),           # bmax - thr = 2^20: the field's largest value is 2^21 - 1
    "full21_bias0": (21, H21 - 1),      # thr = 2^20 - 1: bias 0
    "past21": (21, H21 // 2 - 1),       # bmax - thr = 2^20 + 1: 32-bit fields
    "past21_bias0": (21, H21),          # thr = 2^20: 32-bit fields
    "full32": (32, H32 // 4),           # bmax - thr = 2^31 in a 2-field word
}


def field_patterns(name, lower=0):
    """Three single-strand patterns of length 4 (pids 1, 2, 3: slots 0, 1, 2 of one word).  Slot 0: per column the BEST base scores
    hi, the WORST lo, the THIRD `t` (so that the window T = THIRD[0] WORST[1] WORST[2] BEST[3] scores exactly its min_score where that t lies
    between lo and hi); its
    bmax = 2^20 + 2^19 (21) or 2^31 + 2^29 (32).  Slot 1 scores exactly its min_score on the best window B and min_score + 1 on the
    worst window W; slot 2 hits on B."""
    bits, thr = FIELD_SETS[name]
    span = (H21 + H21 // 2) // 4 if bits == 21 else (H32 + H32 // 4) // 4
    lo = -(span // 2) if bits == 21 else -(span - (1 << 28))
    hi = lo + span
    M = 4 * lo
    ms0 = M + thr
    w0 = np.zeros((4, 4), np.int64)
    for c in range(4):
        w0[c] = [1000 if bits == 21 else 1 << 20] * 4
        w0[c, BEST[c]], w0[c, WORST[c]] = hi, lo
    w0[0, THIRD[0]] = min(max(ms0 - 2 * lo - hi, lo), hi)
    rng = np.random.default_rng(31)
    w1 = rng.integers(-60, 61, (4, 4))
    s1 = lambda x: int(sum(w1[c, x[c]] for c in range(4)))
    w1[0, WORST[0]] += s1(BEST) + 1 - s1(WORST)
    w2 = rng.integers(-60, 61, (4, 4))
    s2 = int(sum(w2[c, BEST[c]] for c in range(4)))
    return [pat(w0, ms0 - lower, 1), pat(w1, s1(BEST) - lower, 2), pat(w2, s2 - 1 - lower, 3)]


def field_region(seed=41):
    """B, W and T planted in the reference and made or broken by SNVs; N sprinkled elsewhere."""
    rng = np.random.default_rng(seed)
    ref = random_bases(rng, 160, n_rate=0.04)
    B, W, T = bases(BEST), bases(WORST), bases([THIRD[0], WORST[1], WORST[2], BEST[3]])
    for at, s in ((10, B), (30, W), (50, T), (70, B), (90, W), (110, "C" + B[1:])):
        ref = put(ref, at, s)
    start = 3000
    recs = [(start + 12, B[2], "T"), (start + 32, W[2], "C"), (start + 110, "C", "A"), (start + 140, ref[140], "N" if ref[140] != "N" else "A")]
    if ref[140] == "N":
        recs = recs[:3]
    recs = [r for r in recs if r[1] != "N"]
    H = 12
    carriers = np.zeros((len(recs), H), bool)
    for v in range(len(recs)):
        carriers[v, rng.choice(H, 4, replace=False)] = True
    return [Region(start, ref, [(start, start + 159), (start + 10, start + 13), (start + 60, start + 75, 2)], recs, carriers)], 6


# ---- thresholds at M - 1, M, M + bmax - 1, M + bmax ------------------------------------------------------------------------------

def threshold_patterns():
    rng = np.random.default_rng(51)
    w = rng.integers(-40, 41, (6, 4))
    w[:, 0], w[:, 1] = -abs(w[:, 0]) - 1, abs(w[:, 1]) + 1  # mixed signs: N is never a column's best or worst base
    base = pat(w, 0, 0)
    M, bmax = plan(base)
    mss = [M - 1, M + bmax // 2, M, M + bmax - 1, M + bmax // 3, M + bmax]
    return [pat(w, ms, pid) for pid, ms in enumerate(mss, 1)], w


def threshold_region():
    pats, w = threshold_patterns()
    best, worst = bases(w.argmax(axis=1)), bases(w.argmin(axis=1))
    rng = np.random.default_rng(52)
    ref = random_bases(rng, 120, n_rate=0.03)
    ref = put(put(put(ref, 20, best), 50, worst), 80, best[:3] + ("A" if best[3] != "A" else "C") + best[4:])
    start = 7000
    recs = [(start + 22, best[2], "ACGT"[(CODE[best[2]] + 1) % 4]), (start + 52, worst[2], "ACGT"[(CODE[worst[2]] + 1) % 4]),
            (start + 83, ref[83], best[3])]
    carriers = np.zeros((3, 8), bool)
    carriers[0, [1, 2]] = carriers[1, [2, 5]] = carriers[2, [0, 5, 6]] = True
    return [Region(start, ref, [(start, start + 119), (start + 18, start + 30)], recs, carriers)], 4


# ---- N as a column's unique best or worst base ----------------------------------------------------------------------------------

POS_COLS, NEG_COLS = [0, 3, 4, 7], [1, 2, 5, 6]  # both halves of the pairs (0,1) (2,3) (4,5) (6,7)


def n_weights():
    rng = np.random.default_rng(61)
    w = np.zeros((8, 4), np.int64)
    for c in range(8):
        w[c] = rng.permutation([1, 2, 3, 4]) * (1 if c in POS_COLS else -1)
    return w


def n_patterns():
    """M = -16, bmax = 32.  Low: min_score M + 1, only windows with N on the positive columns tie or miss.  High: M + bmax - 2, only
    windows with N on the negative columns hit."""
    w = n_weights()
    return [pat(w, -15, 1), pat(w, 14, 2), pat(w, 0, 3)]


def n_windows():
    """(window, N columns) planted: the low pattern's worst window with N on 2, 3, 4 positive columns, the high pattern's best window
    with N on 2, 3, 4 negative columns, odd and even columns alike."""
    w = n_weights()
    lo, hi = w.argmin(axis=1), w.argmax(axis=1)
    out = []
    for src, cols_list in ((lo, [[0, 3], [3, 4, 7], [0, 4, 7], [0, 3, 4, 7]]), (hi, [[1, 5], [1, 2, 6], [2, 5, 6], [1, 2, 5, 6]])):
        for cols in cols_list:
            s = list(bases(src))
            for c in cols:
                s[c] = "N"
            out.append(("".join(s), cols))
    return out


def n_region():
    rng = np.random.default_rng(62)
    ref = random_bases(rng, 40 + 20 * 12)
    start = 12000
    recs, H = [], 10
    for k, (win, cols) in enumerate(n_windows()):
        at = 20 + 20 * k
        if k % 2:  # one of the N bases comes from an ALT allele: the reference has the column's base
            c = cols[-1]
            filled = win[:c] + "ACGT"[k % 4] + win[c + 1:]
            ref = put(ref, at, filled)
            recs.append((start + at + c, filled[c], "N"))
        else:
            ref = put(ref, at, win)
    carriers = np.zeros((len(recs), H), bool)
    for v in range(len(recs)):
        carriers[v, [v % H, (3 * v + 1) % H, (5 * v + 2) % H]] = True
    return [Region(start, ref, [(start, start + len(ref) - 1), (start + 60, start + 140)], recs, carriers)], 5


# ---- every run length and slot count -------------------------------------------------------------------------------------------

def lengths_case(per_length):
    """Lengths 1..32 in one chunk, `per_length` patterns each (1: 32 patterns, 2: 64, 3: 96 = 2, 1, 0 mod 3)."""
    rng = np.random.default_rng(70 + per_length)
    start = 20000
    ref = random_bases(rng, 500, n_rate=0.03)
    pos = sorted(rng.choice(np.arange(5, 480, 6), 24, replace=False))
    recs = []
    for k, p in enumerate(pos):
        b = ref[p]
        if b == "N":
            continue
        alt = "N" if k % 7 == 0 else ("ACGT"[(CODE[b] + 1) % 4] if k % 5 else b + "GA")
        recs.append((start + int(p), b, alt))
    recs.append((start + 485, ref[485], ref[485] + "T") if ref[485] != "N" else (start + 486, ref[486], "C"))
    H = 16
    regions = [Region(start, ref, [(start, start + 499), (start + 100, start + 110), (start + 300, start + 420, 3)], recs,
                      rng.random((len(recs), H)) < 0.3)]
    regions[0].records = [r for r in regions[0].records if r[1] != "N"]
    regions[0].carriers = regions[0].carriers[:len(regions[0].records)]
    pats = []
    for L in range(32, 0, -1):
        for k in range(per_length):
            p = pat(rng.integers(-30, 31, (L, 4)), 0, L)
            if k == 1:
                p = revcomp_pat(p)
            pats.append(p)
    for p in pats:
        p["min_score"] = quantile_threshold(regions, p, 0.85)
    return regions, H // 2, pats


def runs_of(patterns, fields=3):
    """Run lengths G of the triples tables.cpp builds for one chunk holding `patterns` (stable sort by length, longest first)."""
    ls = sorted((len(p["weights"]) for p in patterns if p.get("kind", binding.PATTERN_PWM) == binding.PATTERN_PWM), reverse=True)
    return [(L + 1) // 2 for L in ls[::fields]]


# ---- chunks ------------------------------------------------------------------------------------------------------------------------

def chunk_count(patterns, budget_bytes, fields=3):
    """tables.cpp's greedy split of the ascending pattern_id list into chunks of at most budget_bytes of tables; ranges without a
    PWM are skipped."""
    pids = sorted({p["pattern_id"] for p in patterns})
    by = {q: [p for p in patterns if p["pattern_id"] == q and p.get("kind", binding.PATTERN_PWM) == binding.PATTERN_PWM] for q in pids}
    nbytes = lambda lo, hi: sum(runs_of([p for q in pids[lo:hi] for p in by[q]], fields)) * PAIR_WORDS * 8
    lo, chunks = 0, []
    while lo < len(pids):
        hi = lo + 1
        while hi < len(pids) and nbytes(lo, hi + 1) <= budget_bytes:
            hi += 1
        if any(by[q] for q in pids[lo:hi]):
            chunks.append(pids[lo:hi])
        lo = hi
    return chunks


OTHER = {"kind": binding.PATTERN_OTHER, "min_score": 0}


def chunk_case():
    """table_budget_kb = 8: chunks of one or two pattern ids, OtherPattern-only ids between them, ids 0 and 65535, three and four
    patterns under one id."""
    rng = np.random.default_rng(81)
    start = 30000
    ref = random_bases(rng, 300, n_rate=0.02)
    recs = [(start + p, ref[p], "ACGT"[(CODE[ref[p]] + 2) % 4]) for p in range(7, 290, 23) if ref[p] != "N"]
    H = 12
    regions = [Region(start, ref, [(start, start + 299), (start + 40, start + 60)], recs, rng.random((len(recs), H)) < 0.35)]
    layout = [(0, [32, 32, 31, 30]), (3, None), (7, [32, 30, 28, 5]), (8, None), (9, None), (100, [20, 12]), (101, [32, 32, 31, 3]),
              (4000, [20]), (65534, None), (65535, [32, 31, 28, 8])]
    pats = []
    for pid, lengths in layout:
        if lengths is None:
            pats.append(dict(OTHER, pattern_id=pid))
            continue
        for k, L in enumerate(lengths):
            p = pat(rng.integers(-30, 31, (L, 4)), 0, pid, binding.DIR_N if k % 2 else binding.DIR_P)
            p["min_score"] = quantile_threshold(regions, p, 0.9)
            pats.append(p)
    return regions, H // 2, pats


# ---- sequence, piece and tile ends --------------------------------------------------------------------------------------------------

END_LEN = 10
END_LENGTHS = [END_LEN - 1, END_LEN, END_LEN + 1, 31, 32, 33, 1023, 1024, 1025, 2047, 2048, 2049]


def end_patterns():
    """All-A motifs of length 10: exact (pid 1) and with one mismatch (pid 2, a partial window of nine A's and the N behind the
    sequence's end would score above it), and the exact T motif on the other strand (pid 1)."""
    return [consensus("A" * END_LEN, 0, 1), consensus("A" * END_LEN, 1, 2), consensus("T" * END_LEN, 0, 1, binding.DIR_N)]


def end_regions():
    """Sequences whose last complete window hits, with A's up to the end.  Long ones also hit at starts 127 and 128 (reference
    pieces) and 1023 and 1024 (tiles), and 2047 when the sequence is long enough."""
    rng = np.random.default_rng(91)
    regions, H = [], 8
    for k, n in enumerate(END_LENGTHS):
        start = 40000 + 5000 * k
        ref = random_bases(rng, n, "CGT")
        for a in (127, 1023, 2047):
            if a + 11 + 1 < n - 12:
                ref = put(ref, a - 1, "C" + "A" * 11 + "C")
        ref = ref[:max(0, n - END_LEN)] + "A" * min(n, END_LEN)
        if n > END_LEN:
            ref = put(ref, n - END_LEN - 1, "C")
        recs = []
        if n > 40:
            recs = [(start + 3, ref[3], "A"), (start + n // 2, ref[n // 2], "G" if ref[n // 2] != "G" else "T"), (start + n - 1, "A", "C")]
            if n > 1100:
                recs.insert(1, (start + 130, "A", "G"))
                recs.insert(2, (start + 1020, ref[1020], "A"))
        carriers = np.zeros((len(recs), H), bool)
        for v in range(len(recs)):
            carriers[v, [(v + 1) % H, (2 * v + 3) % H]] = True
        regions.append(Region(start, ref, [(start, start + n - 1), (start + n - 3, start + n - 1)], recs, carriers))
    return regions, H // 2


# ---- configuration windows ------------------------------------------------------------------------------------------------------

LONG, SHORT = "GATTACAGCCTG", "CTG"  # Lmax = 12, a pattern much shorter than it (and the end of it)


def cfg_patterns():
    return [consensus(LONG, 0, 1), consensus(SHORT, 0, 2), consensus(SHORT, 0, 2, binding.DIR_N)]


def mismatch(b):
    return "ACGT"[(CODE[b] + 1) % 4]


def cfg_region():
    """Offsets inside the window (start 50000):
    a: ref LONG and SHORT hits end on the base just before SNV 40 (inherited by its configuration, never scored again);
    b: SNV 80 completes LONG at [69, 80]: the window ends on the first ALT base, starts at 80 - Lmax + 1;
    c: insertion at 120 whose last ALT base starts LONG (the reference bases behind it finish the motif);
    d: deletion at 160 joins LONG across the junction;
    e: SNVs 200 and 211 (Lmax - 2 untouched bases between): LONG at [200, 211] only with both ALTs;
    f: SNVs 240 and 252 (Lmax - 1 untouched bases between): two clusters."""
    rng = np.random.default_rng(101)
    L = len(LONG)
    ref = random_bases(rng, 300, "ACT")
    ref = put(ref, 40 - L, LONG)
    ref = put(ref, 40 - 3, SHORT)
    ref = put(ref, 40, "T")
    ref = put(ref, 69, LONG[:-1] + mismatch(LONG[-1]))
    ref = put(ref, 120, "A" + LONG[1:])
    ref = put(ref, 155, LONG[:6] + "TTT" + LONG[6:])
    ref = put(ref, 200, mismatch(LONG[0]) + LONG[1:-1] + mismatch(LONG[-1]))
    start = 50000
    recs = [(start + 40, "T", "C"), (start + 80, ref[80], LONG[-1]), (start + 120, "A", "A" + "GT" + LONG[0]),
            (start + 160, ref[160:164], ref[160]), (start + 200, ref[200], LONG[0]), (start + 211, ref[211], LONG[-1]),
            (start + 240, ref[240], mismatch(ref[240])), (start + 252, ref[252], mismatch(ref[252]))]
    H = 16
    carriers = np.zeros((len(recs), H), bool)
    for v in range(len(recs)):
        carriers[v, [(3 * v) % H, (3 * v + 1) % H, (5 * v + 7) % H]] = True
    carriers[4:6, [2, 9]] = True  # both SNVs of the cut: a hit only their carriers have
    carriers[4, 12] = carriers[5, 13] = True  # each SNV alone
    carriers[6:8, 14] = True
    inner = [(start, start + 299), (start + 28, start + 39), (start + 66, start + 81, 3), (start + 150, start + 175)]
    return [Region(start, ref, inner, recs, carriers)], H // 2


# ---- long configuration items, many configurations -----------------------------------------------------------------------------

def long_cfg_regions():
    """Region 0: SNVs every 8 bases from offset 42 to 1242, one haplotype carries them all: one configuration whose item starts at
    42 - Lmax + 1 = 31 and spans more than 1,024 starts.  Region 1: 20 SNVs 30 bases apart, 20 single-record configurations and
    more: more than MAX_PIECES = 16 items."""
    rng = np.random.default_rng(111)
    H = 16
    regions = []
    start = 60000
    ref = random_bases(rng, 1400)
    recs = [(start + p, ref[p], mismatch(ref[p])) for p in range(42, 1243, 8)]
    carriers = rng.random((len(recs), H)) < 0.2
    carriers[:, 5] = True
    carriers[:, 6] = False
    regions.append(Region(start, ref, [(start, start + 1399), (start + 500, start + 560)], recs, carriers))
    start = 70000
    ref = random_bases(rng, 700)
    recs = [(start + p, ref[p], mismatch(ref[p])) for p in range(20, 620, 30)]
    carriers = np.zeros((len(recs), H), bool)
    for v in range(len(recs)):
        carriers[v, [v % H, (v + 3) % H]] = True
    regions.append(Region(start, ref, [(start, start + 699)], recs, carriers))
    return regions, H // 2


def long_cfg_patterns(regions):
    rng = np.random.default_rng(112)
    pats = [pat(rng.integers(-30, 31, (12, 4)), 0, 1), pat(rng.integers(-30, 31, (5, 4)), 0, 2)]
    pats.append(revcomp_pat(pats[0]))
    for p in pats:
        p["min_score"] = quantile_threshold(regions, p, 0.9)
    return pats


# ---- inner regions inside a hit ---------------------------------------------------------------------------------------------------

INNER_MOTIF = "TGACCGTAGC"  # L = 10


def inner_region():
    """A reference hit at [h, h + 9] (h = offset 50) that SNV h + 5 destroys (a hit k_cfg_lost takes out), a hit at [g, g + 9]
    (g = offset 150) that SNV g + 4 creates (counted in the configuration's rare path).  Around each: inner regions of 1 and L - 2
    bases strictly inside (not counted), touching the first or the last base (counted), multiplicities 1 and 3."""
    rng = np.random.default_rng(121)
    ref = random_bases(rng, 220)
    ref = put(ref, 50, INNER_MOTIF)
    ref = put(ref, 150, INNER_MOTIF[:4] + mismatch(INNER_MOTIF[4]) + INNER_MOTIF[5:])
    start = 80000
    recs = [(start + 55, INNER_MOTIF[5], mismatch(INNER_MOTIF[5])), (start + 154, ref[154], INNER_MOTIF[4])]
    carriers = np.zeros((2, 12), bool)
    carriers[0, [1, 4, 7]] = carriers[1, [2, 4, 9]] = True
    inner = []
    for h in (start + 50, start + 150):
        inner += [(h + 1, h + 1), (h + 1, h + 8, 3), (h + 4, h + 5, 3), (h, h, 3), (h - 5, h), (h + 9, h + 9, 3), (h + 9, h + 20),
                  (h - 3, h + 12, 3)]
    return [Region(start, ref, inner, recs, carriers)], 6


# ---- the cases ----------------------------------------------------------------------------------------------------------------------

def case(name):
    """(regions, n_samples, patterns, options, scan launches of the full scan or None)."""
    if name in FIELD_SETS:
        regions, S = field_region()
        return regions, S, field_patterns(name), None, 1
    if name == "thresholds":
        regions, S = threshold_region()
        return regions, S, threshold_patterns()[0], None, 1
    if name == "n_columns":
        regions, S = n_region()
        return regions, S, n_patterns(), None, 1
    if name.startswith("lengths"):
        regions, S, pats = lengths_case(int(name[-1]))
        return regions, S, pats, None, 1
    if name == "chunks":
        regions, S, pats = chunk_case()
        return regions, S, pats, {"table_budget_kb": 8}, len(chunk_count(pats, 8 * 1024))
    if name == "ends":
        regions, S = end_regions()
        return regions, S, end_patterns(), None, 1
    if name == "cfg_windows":
        regions, S = cfg_region()
        return regions, S, cfg_patterns(), None, 1
    if name == "long_cfg":
        regions, S = long_cfg_regions()
        return regions, S, long_cfg_patterns(regions), None, 1
    if name == "inner_inside_hit":
        regions, S = inner_region()
        return regions, S, [consensus(INNER_MOTIF, 0, 4)], None, 1
    raise KeyError(name)


CASES = list(FIELD_SETS) + ["thresholds", "n_columns", "lengths1", "lengths2", "lengths3", "chunks", "ends", "cfg_windows", "long_cfg",
                            "inner_inside_hit"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_small_scan_edge(name):
    regions, S, pats, options, launches = case(name)
    check(regions, S, pats, options, launches)


@pytest.mark.gpu
@pytest.mark.parametrize("lower", [0, 1])
def test_small_audit_at_field_boundary(lower):
    """tfbs_audit_block on the exactly-full 21-bit set: its lowered run (every min_score - 1) needs 32-bit fields.  The ties are the
    reference's windows that score exactly min_score; the rows the audit leaves behind are the normal run's.  lower = 1 runs the
    set that starts one below, whose normal run is already in 32-bit fields."""
    regions, S = field_region()
    pats = field_patterns("full21", lower)
    blk = make_block(regions, S)
    ctx = binding.Context(0)
    try:
        ctx.set_option("rows_mode", binding.ROWS_ALL_KEYS)
        ctx.set_patterns(PatternSet(pats))
        ctx.upload_block(blk)
        au = ctx.audit()
        rows = ctx.collect()
    finally:
        ctx.close()
    assert not au["truncated"]
    ref = reference(regions, pats)
    assert np.array_equal(au["hap_group"].reshape(len(regions), -1).astype(np.int64), ref[0]["hap_group"][None, :])
    assert table_rows(au) == reference_hits(regions, pats, tie=True)
    exp = expected_rows(regions, ref, binding.ROWS_ALL_KEYS)
    for k in ("region", "inner", "pattern_id", "vmin", "vmax", "left", "right"):
        assert np.array_equal(np.asarray(rows[k], np.int64), np.asarray(exp[k], np.int64)), "rows after the audit differ in " + k


# ---- each case reaches its edge (CPU) ----------------------------------------------------------------------------------------------

def scores_at(p, seq, i):
    return float(window_scores(np.asarray(seq)[None, i:i + len(p["weights"])], p["weights"])[0, 0])


def test_scan_edges_are_what_they_claim():
    regions, _ = field_region()
    seqs = [seq for _, seq, _ in scanned(regions[0])]
    B = [i for s in seqs for i in range(len(s) - 3) if list(s[i:i + 4]) == BEST]
    assert B
    for name, (bits, thr) in FIELD_SETS.items():
        p0, p1, p2 = field_patterns(name)
        M, bmax = plan(p0)
        assert p0["min_score"] - M == thr and M >= -(1 << 31) and M + bmax < (1 << 31)
        # slot 0 reaches bmax on B, where slot 1 ties and slot 2 hits
        s = seqs[0]
        i = B[0] if B[0] < len(s) - 3 else None
        assert scores_at(p0, s, i) == M + bmax and scores_at(p1, s, i) == p1["min_score"] and scores_at(p2, s, i) > p2["min_score"]
        assert fits(p1, 21) and fits(p2, 21)
        if name in ("full21", "full21_bias0"):
            assert fits(p0, 21) and (bmax - thr == H21 or thr == H21 - 1)
        elif name.startswith("past21"):
            assert not fits(p0, 21) and fits(p0, 32) and (bmax - thr == H21 + 1 or thr == H21)
        else:
            assert not fits(p0, 21) and bmax - thr == H32 and fits(p0, 32) and p0["min_score"] < 0
            assert not fits(dict(p0, min_score=p0["min_score"] - 1), 32)
    # the worst window (score M: a field at 0 with bias 0) and the exact tie of slot 0 are present
    p0 = field_patterns("past21_bias0")[0]
    assert any(scores_at(p0, seqs[0], i) == plan(p0)[0] for i in range(len(seqs[0]) - 3))
    ties = reference_hits(regions, field_patterns("full21"), tie=True)
    assert any(pi == 0 for _, pi, _, _ in ties) and any(pi == 1 for _, pi, _, _ in ties)
    low = field_patterns("full21", 1)
    assert not fits(low[0], 21) and fits(low[0], 32)

    # thresholds: M - 1 always, M ties at the worst window, M + bmax - 1 hits only at the best, M + bmax never
    pats, _ = threshold_patterns()
    regions, _ = threshold_region()
    M, bmax = plan(pats[0])
    assert [p["min_score"] for p in pats[::2]] == [M - 1, M, M + bmax // 3] and [pats[3]["min_score"], pats[5]["min_score"]] == [M + bmax - 1, M + bmax]
    sc = np.concatenate([window_scores(seq[None, :], pats[0]["weights"])[0] for _, seq, _ in scanned(regions[0])])
    assert (sc == M).any() and (sc == M + bmax).any()

    # N: one-sign columns; windows with N on them tie and hit, at even and odd columns
    pats = n_patterns()
    assert plan(pats[0]) == (-16, 32)
    regions, _ = n_region()
    assert any(r[2] == "N" for r in regions[0].records)
    for p in pats[:2]:
        sc = np.concatenate([window_scores(seq[None, :], p["weights"])[0] for _, seq, _ in scanned(regions[0])])
        assert (sc == p["min_score"]).any() and (sc == p["min_score"] + 1).any()
    cols = [c for _, cs in n_windows() for c in cs]
    assert {c % 2 for c in cols if c in POS_COLS} == {0, 1} and {c % 2 for c in cols if c in NEG_COLS} == {0, 1}
    # without N the low pattern always hits and the high one never does: N decides
    w = n_weights()
    assert w.min(axis=1)[POS_COLS].sum() + w.min(axis=1)[NEG_COLS].sum() > -15
    assert w.max(axis=1)[POS_COLS].sum() + w.max(axis=1)[NEG_COLS].sum() < 14

    # every run length, slot counts 0, 1, 2 mod 3, shorter patterns inside longer triples
    for k in (1, 2, 3):
        _, _, pats = lengths_case(k)
        assert sorted({len(p["weights"]) for p in pats}) == list(range(1, 33))
        assert len(pats) % 3 == {1: 2, 2: 1, 3: 0}[k]
        G = runs_of(pats)
        if k == 3:
            assert sorted(set(G)) == list(range(1, 17))  # MAX_RUNS runs
        ls = sorted((len(p["weights"]) for p in pats), reverse=True)
        assert any((ls[t] + 1) // 2 > (ls[t + 2] + 1) // 2 for t in range(0, len(ls) - 2, 3)) or k == 3  # shorter inside longer
        assert sum(G) * PAIR_WORDS * 8 <= 96 * 1024  # one chunk

    # chunks of one or two ids, an OtherPattern-only range between two chunks
    _, _, pats = chunk_case()
    chunks = chunk_count(pats, 8 * 1024)
    pwm_ids = [sorted({p["pattern_id"] for p in pats if "weights" in p and p["pattern_id"] in c}) for c in chunks]
    assert len(chunks) == 4 and {len(c) for c in pwm_ids} == {1, 2}
    assert pwm_ids[0][0] == 0 and pwm_ids[-1][-1] == 65535
    other = [p["pattern_id"] for p in pats if "weights" not in p]
    assert {q for q in other if any(pwm_ids[k][-1] < q < pwm_ids[k + 1][0] for k in range(3))} == {3, 65534}  # between two chunks
    assert max(sum(p["pattern_id"] == q for p in pats) for q in (0, 7, 101, 65535)) >= 4

    # ends: a hit on the last complete window of every sequence at least L long; 127/128 and 1023/1024 starts of one sequence
    regions, _ = end_regions()
    hits = reference_hits(regions, end_patterns())
    for r, reg in enumerate(regions):
        n = len(reg.ref)
        last = {(pi, s - reg.start) for rr, pi, g, s in hits if rr == r and g == 0}
        if n >= END_LEN:
            assert (0, n - END_LEN) in last and (1, n - END_LEN) in last
            tail = reg.codes[n - END_LEN + 1:]
            assert 10 * len(tail) - 10 * (END_LEN - len(tail)) * 0 > end_patterns()[1]["min_score"]  # a partial window would hit
        else:
            assert not last and 10 * n > end_patterns()[1]["min_score"]
        if n > 2000:
            assert {(0, 127), (0, 128), (0, 1023), (0, 1024)} <= last
            assert (0, 2047) in last or n < 2047 + END_LEN + 2
    assert {len(r.ref) for r in regions} == set(END_LENGTHS)

    # configuration windows
    regions, _ = cfg_region()
    reg = regions[0]
    L = len(LONG)
    hits = reference_hits(regions, cfg_patterns())
    ref_hits = {(pi, s - reg.start) for _, pi, g, s in hits if g == 0}
    assert (0, 40 - L) in ref_hits and (1, 40 - 3) in ref_hits  # windows ending on the base before SNV 40
    _, sets = group_haplotypes(reg.carriers)
    gained = {(pi, s - reg.start) for _, pi, g, s in hits if g > 0} - ref_hits
    assert (0, 80 - L + 1) in gained  # ends on SNV 80's ALT base
    assert (0, 120) in gained  # starts on the insertion's last ALT base (positions: every ALT base at 120)
    assert (0, 155) in gained  # straddles the deletion's junction
    assert (0, 200) in gained
    both = [g for g, s in enumerate(sets, 1) if {4, 5} <= set(s)]
    assert both and all((0, 200) in {(pi, x - reg.start) for _, pi, gg, x in hits if gg == g} for g in both)
    for v in (4, 5):
        alone = [g for g, s in enumerate(sets, 1) if v in s and {4, 5} - {v} - set(s)]
        assert alone and not any(pi == 0 and x - reg.start == 200 and gg in alone for _, pi, gg, x in hits)
    gap = lambda a, b: reg.records[b][0] - reg.records[a][0] - 1
    assert gap(4, 5) == L - 2 and gap(6, 7) == L - 1

    # long configuration item at p0 % 32 == 31 over more than 1,024 starts; more than 16 configurations
    regions, _ = long_cfg_regions()
    r0 = regions[0]
    first, last = r0.records[0][0] - r0.start, r0.records[-1][0] - r0.start
    assert all(b[0] - a[0] < L for a, b in zip(r0.records, r0.records[1:]))
    p0 = first - L + 1
    assert p0 % 32 == 31 and last - p0 + 1 > 1024 and r0.carriers[:, 5].all()
    assert len(regions[1].records) > 16 and all(b[0] - a[0] > L for a, b in zip(regions[1].records, regions[1].records[1:]))

    # inner regions strictly inside a hit are not counted, touching ones are; on a lost and on a gained hit
    regions, _ = inner_region()
    reg = regions[0]
    e = reference(regions, [consensus(INNER_MOTIF, 0, 4)])[0]
    hg, counts = e["hap_group"], e["counts"]
    g_lost = hg[1]  # carries SNV h + 5 only
    g_gain = hg[2]  # carries SNV g + 4 only
    for base, row in ((0, counts[0]), (8, counts[g_gain])):
        assert list(row[base:base + 8]) == [0, 0, 0, 3, 1, 3, 1, 3]
    assert list(counts[g_lost][:8]) == [0] * 8 and list(counts[0][8:]) == [0] * 8
    assert sum(1 for x in reg.mult if x == 3) >= 4 and max(b - a + 1 for a, b in reg.inner[:3]) == len(INNER_MOTIF) - 2


def test_scan_edges_on_emulated_kernels():
    """The GPU tests named *small* on tests/cuda_emu/libtfbs_emu.so (the product's kernel sources on a CUDA-on-host shim)."""
    import subprocess
    from test_large_regions import EMU, run_marked_gpu_tests
    subprocess.check_call(["make", "-C", EMU, "-j2", "libtfbs_emu.so"], stdout=subprocess.DEVNULL)
    env = dict(os.environ, TFBS_B200_LIB=os.path.join(EMU, "libtfbs_emu.so"))
    out = run_marked_gpu_tests(env, "tests/test_scan_edges.py", "small")
    assert "%d passed" % (len(CASES) + 2) in out
