/*
 * tfbs.h -- C ABI of the B200-native find-tfbs hot path.
 *
 * This header is the drop-in boundary for the reference's per-region pipeline
 * (all citations are paths under the reference repository, Helkafen/find-tfbs):
 *
 *   find_all_matches          src/main.rs:94-154      (haplotype build + PWM scan)
 *     load_haplotypes         src/haplotype.rs:77-88
 *     patch_haplotype         src/haplotype.rs:94-156
 *     matches / apply_pwm     src/pattern.rs:119-171
 *   count_matches_by_sample   src/main.rs:500-534
 *   counts_as_genotypes       src/main.rs:439-458     (v = l + r, min == max filter)
 *
 * The reference has no FFI of its own; the seam is the Rust call sequence inside
 * process_peak (src/main.rs:409-420).  A Rust driver would bind these entry points
 * with bindgen and feed one tfbs_block per chunk of merged regions (the reference
 * hands out chunks of 50 regions, src/main.rs:375-381).  See INTEGRATION.md.
 *
 * Plain C only: fixed-width integers, pointers and sizes.  No C++ or torch types.
 */
#ifndef TFBS_H
#define TFBS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TFBS_ABI_VERSION 2

/* Nucleotide codes: enum Nucleotide { A, C, G, T, N } (src/types.rs:5-8). */
enum { TFBS_NUC_A = 0, TFBS_NUC_C = 1, TFBS_NUC_G = 2, TFBS_NUC_T = 3, TFBS_NUC_N = 4 };

/* enum Pattern { PWM{..}, OtherPattern{..} } (src/types.rs:86-90). */
enum { TFBS_PATTERN_PWM = 0, TFBS_PATTERN_OTHER = 1 };
/* enum PWMDirection { P, N } (src/types.rs:72-75). */
enum { TFBS_DIR_P = 0, TFBS_DIR_N = 1 };

/* Status codes (negative = the condition on which the reference panics). */
enum {
    TFBS_OK = 0,
    TFBS_ERR_INVALID_ARGUMENT = -1,
    TFBS_ERR_CUDA = -2,              /* CUDA runtime failure or no usable device */
    TFBS_ERR_UNKNOWN_NUCLEOTIDE = -3,/* util.rs:15 "Unknown nucleotide" */
    TFBS_ERR_REF_MISMATCH = -4,      /* haplotype.rs:126-128 */
    TFBS_ERR_MISSING_CASE = -5,      /* haplotype.rs:141-143 "Missing case in haplotype patcher" */
    TFBS_ERR_SCORE_RANGE = -6,       /* weights too large for exact 32-bit scoring */
    TFBS_ERR_STATE = -7,             /* call order violated (e.g. collect before submit) */
    TFBS_ERR_INTERNAL = -8           /* hash collision retry exhausted etc. */
};

/*
 * One pattern, laid out as the reference holds it: Pattern::PWM { weights, name, pattern_id,
 * min_score, direction } with Weight { acgtn: [a, c, g, t, 0] } (src/types.rs:86-113).
 * Forward (P) and reverse-complement (N) patterns are separate entries that share
 * pattern_id (src/pattern.rs:73-77); the caller passes them exactly as parse_pwm_files
 * would have produced them.  A window scores sum_c weights[c][nuc(i+c)] with N -> 0 and
 * is a hit iff score > min_score (src/pattern.rs:125-129,151).
 */
typedef struct tfbs_pattern {
    const int32_t* weights; /* len x 4, row-major [column][A,C,G,T]; may be NULL if kind != PWM */
    uint32_t len;           /* pattern_length(); 0 for OtherPattern (src/types.rs:92-101) */
    int32_t min_score;
    uint16_t pattern_id;
    uint8_t direction;      /* TFBS_DIR_* (informational) */
    uint8_t kind;           /* TFBS_PATTERN_*; OtherPattern never matches (src/pattern.rs:166-168) */
} tfbs_pattern;

/*
 * One original BED region that select_inner_peaks (src/main.rs:62-72) attached to a merged
 * region.  `multiplicity` is how many times the identical (bed, start, end) occurs in that
 * BED file: the reference visits such a region once per occurrence and so multiplies its
 * counts (src/main.rs:503-505).  Use 1 unless the BED file holds duplicates.
 */
typedef struct tfbs_inner_region {
    int64_t start;          /* inclusive, 0-based (src/bed.rs:15) */
    int64_t end;            /* inclusive */
    uint32_t bed_index;     /* which BED file (caller-defined numbering) */
    uint32_t multiplicity;
} tfbs_inner_region;

/*
 * One biallelic record returned by the BCF fetch of a region's extended window
 * (src/haplotype.rs:16-28), i.e. a Diff { pos, reference, alternative } (src/types.rs:39-44)
 * plus the row of the carrier bit matrix that says which haplotypes carry ALT.
 */
typedef struct tfbs_variant {
    int64_t pos;            /* 0-based record.pos() */
    uint32_t ref_off;       /* REF allele: allele_bases[ref_off .. ref_off + ref_len) */
    uint32_t ref_len;
    uint32_t alt_off;       /* ALT allele */
    uint32_t alt_len;
    uint32_t carrier_row;   /* row of tfbs_block.carriers */
    uint32_t reserved;
} tfbs_variant;

/*
 * A block of merged regions with everything process_peak (src/main.rs:395-436) reads for
 * them.  Haplotype index h = 2 * sample_id + side, side 0 = Left, 1 = Right
 * (src/types.rs:29-30,66-70); sample_id indexes the *selected* samples (src/main.rs:293-313).
 * Bit h of carrier row v is set iff the reference's load_diffs would push that Diff for h:
 * left iff the first GT value is Unphased(1), right iff the second is Phased(1)
 * (src/haplotype.rs:34-49).
 */
typedef struct tfbs_block {
    uint32_t n_regions;
    uint32_t n_samples;
    const int64_t* region_start;   /* [n_regions] extended window start = merged.start - Lmax + 1 (main.rs:407) */
    const int64_t* region_end;     /* [n_regions] extended window end   = merged.end + Lmax - 1, inclusive */
    const uint64_t* ref_off;       /* [n_regions + 1] window r = ref_bases[ref_off[r] .. ref_off[r+1]) */
    const uint8_t* ref_bases;      /* ASCII ACGTNacgtn as read from the FASTA (util.rs:4-16); base i of a
                                      window has pos = region_start + i (util.rs:22-31).  A window may be
                                      shorter than region_end - region_start + 1 (haplotype.rs:183-185). */
    const uint32_t* inner_off;     /* [n_regions + 1] */
    const tfbs_inner_region* inner;/* inner regions per merged region */
    const uint32_t* var_off;       /* [n_regions + 1] */
    const tfbs_variant* variants;  /* per region, in BCF record order */
    const uint8_t* allele_bases;   /* ASCII */
    uint64_t allele_bytes;
    const uint32_t* carriers;      /* [n_carrier_rows][carrier_pitch] little-endian bit h -> word h/32, bit h%32 */
    uint32_t n_carrier_rows;
    uint32_t carrier_pitch;        /* 32-bit words per row, >= ceil(2 * n_samples / 32) */
} tfbs_block;

/*
 * Result rows: one per key (merged region, inner region, pattern_id) of
 * count_matches_by_sample (src/main.rs:500-534) that survives the filter.  left/right are the
 * reference's (Vec<u32>, Vec<u32>) value.  Rows come in a deterministic order: by region,
 * then pattern_id ascending, then inner index.  Pointers stay valid until the next
 * tfbs_collect / tfbs_collect_grouped, the second-next tfbs_submit_block / tfbs_run_resident, or tfbs_destroy on the same context.
 */
typedef struct tfbs_rows {
    uint64_t n_rows;
    uint32_t n_samples;
    uint32_t count_bytes;          /* size of one element of left / right: 4 (uint32_t) unless option "rows_width" = 0 let the
                                      library return the narrowest type that holds every count of the block (1, 2 or 4) */
    const uint32_t* region;        /* [n_rows] index of the merged region inside the block */
    const uint32_t* inner;         /* [n_rows] index into tfbs_block.inner */
    const uint16_t* pattern_id;    /* [n_rows] */
    const uint32_t* vmin;          /* [n_rows] min over samples of left + right (main.rs:450) */
    const uint32_t* vmax;          /* [n_rows] max over samples of left + right (main.rs:451) */
    const uint32_t* left;          /* [n_rows * n_samples] elements of count_bytes bytes (uint32_t by default) */
    const uint32_t* right;         /* [n_rows * n_samples] */
} tfbs_rows;

/*
 * The same rows with identical count vectors stored once ("grouped rows"): haplotypes that carry the same records in a region
 * (group_by_diffs, src/haplotype.rs:65-75) have the same count for every key, so a row holds one count per GROUP of the region and
 * the haplotype -> group map is returned once per region.  A sample's (left, right) of count_matches_by_sample (src/main.rs:500-534)
 * is (count[hap_group[2 * sample]], count[hap_group[2 * sample + 1]]); tfbs_expand_rows does exactly that.  Counts are packed as
 * `bits`-wide offsets from the row's smallest count (bits = 0: every group has the count `base`).  This is what crosses PCIe for
 * large cohorts: about 1/10 of the dense rows.
 */
typedef struct tfbs_grouped_rows {
    uint64_t n_rows;
    uint32_t n_samples;
    uint32_t n_regions;
    const uint32_t* region;        /* [n_rows] as in tfbs_rows */
    const uint32_t* inner;         /* [n_rows] */
    const uint16_t* pattern_id;    /* [n_rows] */
    const uint32_t* vmin;          /* [n_rows] */
    const uint32_t* vmax;          /* [n_rows] */
    const uint32_t* base;          /* [n_rows] smallest per-haplotype count of the row */
    const uint8_t* bits;           /* [n_rows] width of a packed entry: 0, 1, 2, 4, 8, 16 or 32 */
    const uint64_t* offset;        /* [n_rows] first 32-bit word of the row in `packed` */
    const uint32_t* packed;        /* per row ceil(n_groups[region] * bits / 32) words, little-endian bit order: entry g = count of
                                      group g minus base, at bits [g * bits, (g + 1) * bits) of the row */
    uint64_t packed_words;
    const uint32_t* n_groups;      /* [n_regions] distinct haplotypes of the region incl. the reference haplotype (group 0) */
    const void* hap_group;         /* [n_regions * 2 * n_samples] group of haplotype h = 2 * sample + side in its region, as uint16_t
                                      or uint32_t (hap_group_bytes); 0 = the reference haplotype (main.rs:103-105,129-131), the
                                      other groups numbered 1.. in order of their smallest haplotype */
    uint32_t hap_group_bytes;      /* 2 or 4 */
    uint32_t reserved;
} tfbs_grouped_rows;

/* Individual hits (struct Match, src/types.rs:32-37), for debugging and parity tests. */
typedef struct tfbs_matches {
    uint64_t n_matches;
    const uint32_t* region;        /* [n_matches] */
    const uint32_t* pattern_index; /* [n_matches] index into the array given to tfbs_set_patterns */
    const uint32_t* group;         /* [n_matches] distinct-haplotype group inside the region, 0 = reference */
    const int64_t* start;          /* [n_matches] range.start = pos of the window's first base (pattern.rs:156) */
    /* carrier lists: group of haplotype h in region r is hap_group[r * 2 * n_samples + h] */
    const uint32_t* hap_group;
    uint32_t n_samples;
    uint32_t truncated;            /* 1 if the match buffer overflowed (n_matches is then a lower bound) */
} tfbs_matches;

/*
 * Audit of one block (tfbs_audit_block): everything about it that the reference leaves undefined or that sits exactly on a
 * threshold, so that a bit-exact comparison can enumerate those places instead of tripping over them.
 *   ties       windows whose score EQUALS min_score.  They are not hits (pattern.rs:151 is a strict >), but they are the windows
 *              a +-1 difference in a weight or threshold (f32 parsing, pattern.rs:13-16) would flip.  Same tuple as a match.
 *   hap_flags  per (region, haplotype): TFBS_HAP_TRUNCATED = its diff list ran into the truncation exit of patch_haplotype
 *              (overlapping variants, haplotype.rs:144-149); TFBS_HAP_OVERWRITTEN = its diff list patched to the same
 *              (nuc, pos) vector as another one's, its entry of the sequence-keyed map was overwritten (haplotype.rs:84) and it is
 *              counted with the reference haplotype (main.rs:103-105,129-131).  Which of the colliding lists survives depends on
 *              HashMap order in the reference ("reference undefined"); here the one with the smallest first haplotype does.
 */
enum { TFBS_HAP_TRUNCATED = 1, TFBS_HAP_OVERWRITTEN = 2 };
typedef struct tfbs_audit {
    uint64_t n_ties;
    const uint32_t* tie_region;        /* [n_ties] */
    const uint32_t* tie_pattern_index; /* [n_ties] index into the array given to tfbs_set_patterns */
    const uint32_t* tie_group;         /* [n_ties] group inside the region (hap_group numbering), 0 = reference */
    const int64_t* tie_start;          /* [n_ties] pos of the window's first base */
    const uint32_t* hap_group;         /* [n_regions * 2 * n_samples] */
    const uint8_t* hap_flags;          /* [n_regions * 2 * n_samples] TFBS_HAP_* bits */
    uint32_t n_regions;
    uint32_t n_samples;
    uint32_t truncated;                /* 1 if the hits did not fit even into the enlarged match buffer (> 2^31): the tie list is incomplete */
    uint32_t reserved;
} tfbs_audit;

/*
 * Attribution of one block's rows (option "attribution" = 1, default path only; tfbs_get_attribution): which CONFIGURATIONS -- the
 * records of one cluster of nearby records that a haplotype carries together -- change each row's count, and by how much.  For row j
 * (row j of the tfbs_collect / tfbs_collect_grouped that returned the block) and every haplotype h of its region, the count h gets
 * (left or right) is exactly
 *     ref_count[j] + sum of term_diff[t] over t in [term_off[j], term_off[j + 1]) with term_cfg[t] in the list of group(h)
 * where group(h) = hap_group of h in its region and the list of group g of region r is group_cfg[group_cfg_off[G] ..
 * group_cfg_off[G + 1]), G = (sum of n_groups over the regions before r) + g.  Counts are integers: the equality has no tolerance.
 * Configuration ids are numbered block-wide, by region, then by their first carrier group and position: they do not depend on hash
 * seeds or on the order threads ran in.
 */
enum { TFBS_CFG_TRUNCATES = 1 };
typedef struct tfbs_attribution {
    uint64_t n_rows;               /* == n_rows of the collect */
    const uint32_t* ref_count;     /* [n_rows] count of the region's reference haplotype for the row's key */
    const uint64_t* term_off;      /* [n_rows + 1] */
    const uint32_t* term_cfg;      /* [term_off[n_rows]] configurations whose count difference for the key is not 0, ascending */
    const int32_t* term_diff;      /* [term_off[n_rows]] the configuration's count minus the reference haplotype's count */
    uint64_t n_cfgs;               /* configurations of the block */
    const uint32_t* cfg_region;    /* [n_cfgs] merged region of the configuration */
    const uint8_t* cfg_flags;      /* [n_cfgs] TFBS_CFG_TRUNCATES: its walk reached patch_haplotype's truncation exit (haplotype.rs:144-149),
                                      its difference includes the reference hits lost behind it */
    const uint64_t* cfg_rec_off;   /* [n_cfgs + 1] */
    const uint32_t* cfg_rec;       /* records of the configuration as indices into tfbs_block.variants, in the order the walk applies
                                      them (position order) */
    uint64_t n_groups_total;       /* sum of n_groups over the regions */
    const uint64_t* group_cfg_off; /* [n_groups_total + 1] */
    const uint32_t* group_cfg;     /* configurations whose difference the group's count includes, in the order of the group's records.
                                      Empty for group 0 and for groups overwritten in the sequence-keyed map (counted as the reference
                                      haplotype); behind a truncation only what the haplotype still applies */
} tfbs_attribution;

/*
 * Binding sites behind the attribution's terms (option "sites" = 1 together with "attribution" = 1; tfbs_get_sites).  For
 * configuration c (the ids of tfbs_attribution) take two multisets of (pattern_index, start, score) hit triples: A, the hits of the
 * region's extended window patched with c's records alone (truncation exit included), and R, the hits of the unpatched window.  A hit
 * is a complete window with score > min_score; start is the position of its first base (pattern.rs:156: bases an insertion adds share
 * its anchor's position).  The sites of c are A - R with change +1 (gained) and R - A with change -1 (lost), multiset differences: a
 * hit that survives unchanged is not listed, one whose score moves but stays above the threshold is a lost / gained pair.  For every
 * row j with pattern_id p and inner region k, multiplicity(k) times the sum of change over c's sites whose pattern has id p and whose
 * range [start, start + L - 1] overlaps k (range.rs:18-21) is c's term_diff for row j, or 0 when c has no term there.
 * Sites are ordered by configuration, then by (pattern_index, start, score, change) ascending; they do not depend on hash seeds, on
 * the order threads ran in or on the stream the block ran on.
 */
typedef struct tfbs_sites {
    uint64_t n_cfgs;                /* == tfbs_attribution.n_cfgs of the same collect */
    const uint64_t* site_off;       /* [n_cfgs + 1]: sites of configuration c are [site_off[c], site_off[c + 1]) */
    const uint32_t* pattern_index;  /* index into the array given to tfbs_set_patterns (gives pattern_id, strand, L) */
    const int64_t* start;           /* as tfbs_matches.start */
    const int32_t* score;           /* exact window score */
    const int8_t* change;           /* +1 gained, -1 lost */
} tfbs_sites;

/*
 * Binding sites of every record on its own (option "record_sites" = 1; tfbs_get_record_sites).  Let record v be
 * tfbs_block.variants[v], in region r, and take two multisets of (pattern_index, start, score) hit triples: A, the hits of r's extended
 * window patched with v alone, and R, the hits of the unpatched window -- the definition of tfbs_sites with the configuration replaced
 * by the single record.  The sites of v are A - R with change +1 and R - A with change -1, ordered within a record by (pattern_index,
 * start, score, change) ascending.  They do not depend on hash seeds, the order threads ran in, the stream the block ran on, the
 * fan-out or on who carries v: a record no selected sample carries has its sites too.
 * A record with a flag has no sites:
 *   TFBS_REC_OUTSIDE        pos lies outside the region's extended window: patch_haplotype never applies it (haplotype.rs:95);
 *   TFBS_REC_REF_MISMATCH   patch_haplotype would panic on a haplotype that carries only v: REF does not match (haplotype.rs:126-128);
 *   TFBS_REC_MISSING_CASE   ... or a multi-base REF and ALT (haplotype.rs:141-143).
 * A record some haplotype carries fails the block with TFBS_ERR_REF_MISMATCH / TFBS_ERR_MISSING_CASE as always, so only records nobody
 * carries show the last two flags.  A record alone never reaches the truncation exit.
 */
enum { TFBS_REC_OUTSIDE = 1, TFBS_REC_REF_MISMATCH = 2, TFBS_REC_MISSING_CASE = 4 };
typedef struct tfbs_record_sites {
    uint64_t n_records;             /* == var_off[n_regions] of the block: every record, in tfbs_block.variants order */
    const uint8_t* rec_flags;       /* [n_records] TFBS_REC_* */
    const uint64_t* site_off;       /* [n_records + 1]: sites of record v are [site_off[v], site_off[v + 1]) */
    const uint32_t* pattern_index;  /* as tfbs_sites */
    const int64_t* start;
    const int32_t* score;
    const int8_t* change;
} tfbs_record_sites;

/* Row filter: which keys tfbs_collect returns. */
enum {
    TFBS_ROWS_VARYING = 0, /* only keys with min != max, i.e. those counts_as_genotypes keeps (main.rs:456-458) */
    TFBS_ROWS_ALL_KEYS = 1 /* every key count_matches_by_sample creates (>= 1 hit, main.rs:517-528) */
};

/* Per-stage device timings and work counters of the most recent run. */
typedef struct tfbs_stats {
    uint64_t n_regions;
    uint64_t n_groups;          /* distinct haplotype sequences scanned, incl. one reference per region */
    uint64_t executed_cells;    /* sum over scanned (group, pattern) of max(0, len - L + 1) * L */
    uint64_t nominal_cells;     /* the same sum over every haplotype of every sample (2 * n_samples per region) */
    uint64_t n_hits;            /* above-threshold windows over all scanned groups */
    uint64_t n_keys;            /* candidate (region, inner, pattern_id) keys */
    uint64_t n_rows;
    uint64_t h2d_bytes;
    uint64_t d2h_bytes;
    uint32_t scan_launches;     /* launches of the PWM scan kernel */
    uint32_t total_launches;    /* all kernel launches of the run */
    float ms_group;             /* K0: signature hash + grouping */
    float ms_build;             /* K1: haplotype build */
    float ms_scan;              /* K2: work list, packing of the scored bases, PWM scan, finish (sum over batches) */
    float ms_count;             /* K3: fan-out, filter, row compaction */
    float ms_total;             /* first launch to last, device time */
    uint32_t sm_count;
    uint32_t scan_ctas;
    uint64_t evaluated_cells;   /* cells the scan kernel really scored: == executed_cells without delta scoring, less with it */
    uint64_t n_scan_items;      /* ranges of window starts handed to the scan kernel */
    float ms_scan_kernel;       /* device time of the k_scan launches alone (CUDA events around them), summed over batches */
    uint32_t n_dropped;         /* groups overwritten in the sequence-keyed map (haplotype.rs:84; SURVEY A.6 Q4) */
    uint32_t n_truncated;       /* haplotypes truncated by an overlapping variant (haplotype.rs:144-149) */
    uint32_t reserved;          /* default path: keys for which the per-group count vector had to be built (the others have the
                                   reference haplotype's count for everybody) */
    uint64_t scan_input_bytes;  /* algorithmic HBM bytes the scan launches read: 12 B per 32 packed bases (2 bit + N mask) of every
                                   scored entry, once per pattern chunk, plus the chunk's tables once per CTA */
} tfbs_stats;

typedef struct tfbs_ctx tfbs_ctx;

/* Library / ABI version; never touches CUDA. */
int tfbs_abi_version(void);

/* Create a context on CUDA device `device`.  Fails (TFBS_ERR_CUDA) when no device is usable:
 * there is no CPU fallback. */
int tfbs_create(int device, tfbs_ctx** out);
void tfbs_destroy(tfbs_ctx* ctx);

/* Message of the last failing call on this context ("" if none); for ctx == NULL the message
 * of the last failing tfbs_create of the calling thread.  Mirrors the reference's panic text. */
const char* tfbs_last_error(const tfbs_ctx* ctx);

/* Options: "rows_mode" (TFBS_ROWS_*), "record_matches" (0/1), "max_matches" (capacity of the
 * match buffer), "verify_groups" (0/1, exact check of hash-grouped haplotypes, default 1),
 * "scan_format" (0 auto, 1 force 32-bit tables), "delta" (default 1: score a patched haplotype only where its windows
 * touch a variant and inherit every other hit from the region's reference haplotype -- exact, scores are integers; 0: score
 * every distinct haplotype in full like the reference does; forced to 0 while "record_matches" is on), "scratch_mb" (upper bound of
 * the device scratch a block may use; a block that needs more fails with TFBS_ERR_INVALID_ARGUMENT: submit fewer regions at a time),
 * "table_budget_kb", "rows_width" (32 = counts come back as uint32_t, the reference's Vec<u32>; 0 = the narrowest of 8/16/32 bits
 * that holds every count of the block, see tfbs_rows.count_bytes -- result rows are the dominant PCIe traffic of large cohorts),
 * "fan_vector" (0 = automatic, the default: the fan-out keeps its per-group count vectors in shared memory and switches to device
 * memory when a region of the block may have more distinct haplotypes than shared memory holds, 53,120; 1 = always in device
 * memory, for tests -- results are the same either way), "region_tables" (1 = the default: the default path groups the haplotypes
 * of a region in one CTA's shared memory when the block's haplotypes and records per region fit there, and with the block-wide
 * tables otherwise; 0 = always the block-wide tables, for tests and comparisons -- results are the same either way), "attribution" (0 = off, the default; 1 = the default path also keeps the
 * per-row count differences of every configuration for tfbs_get_attribution: the rows themselves do not change), "sites" (0 = off,
 * the default; 1 = the default path also keeps the hits each configuration gains and loses, with their exact scores, for
 * tfbs_get_sites; needs "attribution" = 1, else tfbs_submit_block / tfbs_run_resident fail with TFBS_ERR_INVALID_ARGUMENT),
 * "record_sites" (0 = off, the default; 1 = the default path also scores every record of the block alone and keeps its sites for
 * tfbs_get_record_sites, independently of "attribution" and "sites"; a block with regions but no sample fails with
 * TFBS_ERR_INVALID_ARGUMENT), "dual_stream"
 * (0 = off, the default; 1 = consecutive blocks of the default scoring mode alternate between two lanes, each with its own kernel
 * and copy streams and its own device scratch, so that the kernels of the two blocks in flight overlap on the device: worth it when
 * blocks are small, while a second lane doubles the scratch of large blocks; fails with TFBS_ERR_STATE while blocks are in flight). */
int tfbs_set_option(tfbs_ctx* ctx, const char* key, int64_t value);

/* Replace the pattern list (the reference's pwm_list, src/main.rs:237). */
int tfbs_set_patterns(tfbs_ctx* ctx, const tfbs_pattern* patterns, uint32_t n_patterns);

/* Host-buffer path: enqueue the copy of the block to the device and the whole pipeline, then return -- nothing is waited for
 * (default scoring mode; with "delta" = 0 or "record_matches" the call runs the block to completion).  Up to TWO blocks may be in
 * flight per context: the copies of block i + 1 overlap the kernels of block i, the rows of block i travel back while block i + 1
 * is computed.  A third tfbs_submit_block before a tfbs_collect fails with TFBS_ERR_STATE.  The caller's buffers must stay valid and
 * unchanged until the tfbs_collect that returns this block's rows (they are read by asynchronous copies when page-locked). */
int tfbs_submit_block(tfbs_ctx* ctx, const tfbs_block* block);

/* Wait for the OLDEST block in flight -- the only place the host waits for the device -- and expose its rows as the reference's
 * (left, right) vectors (expanded on the device, then copied). */
int tfbs_collect(tfbs_ctx* ctx, tfbs_rows* out);

/* Same, but the rows come back grouped (see tfbs_grouped_rows): the compact form for large cohorts.  Default scoring mode only. */
int tfbs_collect_grouped(tfbs_ctx* ctx, tfbs_grouped_rows* out);

/*
 * Result arena: caller-owned host memory that receives the grouped rows of every block DIRECTLY by the device -> host copies, e.g. a
 * POSIX shared-memory segment that the process owning the VCF writer has mapped: with one process per GPU this is how the rows of
 * all GPUs are gathered on one host without a collective (regions are independent, src/main.rs:395-429).  The library page-locks the
 * memory.  It is used as two halves of bytes / 2 (blocks in flight alternate, first block -> first half); each half starts with a
 * tfbs_arena_header, every array sits at the byte offset the header gives (relative to the header) and has the layout of the
 * tfbs_grouped_rows member of the same name.  `sequence` is written last, after the copies have completed: a reader that sees it
 * change finds a complete block.  tfbs_collect_grouped fails with TFBS_ERR_INVALID_ARGUMENT when a block does not fit its half.
 * base == NULL goes back to the library's own buffers.
 */
#define TFBS_ARENA_MAGIC 0x3152415342465400ULL /* "\0TFBSAR1" */
typedef struct tfbs_arena_header {
    uint64_t magic;
    uint64_t sequence;         /* number of blocks this half has received */
    uint64_t n_rows;
    uint64_t packed_words;
    uint32_t n_samples;
    uint32_t n_regions;
    uint32_t hap_group_bytes;
    uint32_t reserved;
    uint64_t off_region, off_inner, off_pattern_id, off_vmin, off_vmax, off_base, off_bits, off_offset, off_packed, off_n_groups,
        off_hap_group;
    uint64_t bytes_used;       /* header + arrays */
} tfbs_arena_header;
int tfbs_set_result_arena(tfbs_ctx* ctx, void* base, size_t bytes);

/* Host side of grouped rows: (left, right) of rows [first_row, first_row + n_rows), n_rows * n_samples uint32_t each.  Pure host
 * code, no CUDA call; thread-safe. */
int tfbs_expand_rows(const tfbs_grouped_rows* rows, uint64_t first_row, uint64_t n_rows, uint32_t* left, uint32_t* right);

/*
 * Sample-block sharding (the secondary partition for biobank-scale cohorts, BASELINE.json configs[3]): the same regions and patterns
 * are run once per block of samples, on any GPU, with "rows_mode" = TFBS_ROWS_ALL_KEYS.  Counts are per sample, so the blocks'
 * rows concatenate along the sample axis; the min != max filter of counts_as_genotypes (src/main.rs:450-458) needs ALL samples and
 * is applied by this call after the gather.  parts[p] = the grouped rows of sample block p.  For every key that survives, in row
 * order: region / inner / pattern_id, vmin / vmax over all samples, and part_row[p * cap + j] = its row in parts[p], or UINT64_MAX
 * when block p had no hit for the key (every sample of the block counts 0, src/main.rs:517-528); expand block p's share of row j with
 * tfbs_expand_rows(parts[p], part_row[p * cap + j], 1, ...).  *n_out = surviving keys; when it exceeds `cap` only the first `cap`
 * were written (call with cap = 0 and NULL arrays to size them).  Pure host code, no CUDA call; thread-safe.
 */
int tfbs_merge_sample_blocks(const tfbs_grouped_rows* const* parts, uint32_t n_parts, uint64_t cap, uint32_t* region, uint32_t* inner,
                             uint16_t* pattern_id, uint32_t* vmin, uint32_t* vmax, uint64_t* part_row, uint64_t* n_out);

/*
 * Merged regions of all BED files on the device: load_peak_files' RangeStack (src/bed.rs:37-45, src/range.rs:43-87) -- the ranges
 * sorted by start (stable) and folded from the left with Range::overlaps / Range::merge (range.rs:18-36) -- as a stable rank, a
 * prefix maximum of the ends and a compaction.  start / end: the concatenated inclusive ranges of every BED file (bed.rs:15);
 * out_start / out_end: room for n ranges; *n_out = merged ranges, ascending by start (bed.rs:40-44).  A range with end < start
 * fails with TFBS_ERR_INVALID_ARGUMENT (the fold is then order-dependent; fold such input on the host with the literal rule).
 * Synchronous; independent of the blocks in flight.
 */
int tfbs_merge_regions(tfbs_ctx* ctx, const uint64_t* start, const uint64_t* end, uint64_t n, uint64_t* out_start, uint64_t* out_end,
                       uint64_t* n_out);

/* Attribution (see tfbs_attribution) of the block the last tfbs_collect or tfbs_collect_grouped returned; both forms give the same
 * rows in the same order.  That collect already copied it to the host (option "attribution" on for the run), so blocks submitted
 * since do not affect it.  Fails with TFBS_ERR_STATE when nothing has been collected, when option "attribution" was off for that run,
 * or when the run was a full scan ("delta" = 0 or "record_matches").  Pointers stay valid as those of tfbs_rows do. */
int tfbs_get_attribution(tfbs_ctx* ctx, tfbs_attribution* out);

/* Sites (see tfbs_sites) of the block the last tfbs_collect or tfbs_collect_grouped returned, copied to the host by that collect
 * right after its attribution.  Fails with TFBS_ERR_STATE when nothing has been collected, when option "sites" was off for that run,
 * or when the run was a full scan ("delta" = 0, "record_matches" or the audit).  Pointers stay valid as those of tfbs_rows do. */
int tfbs_get_sites(tfbs_ctx* ctx, tfbs_sites* out);

/* Record sites (see tfbs_record_sites) of the block the last tfbs_collect or tfbs_collect_grouped returned, copied to the host by that
 * collect behind its attribution and sites.  Fails with TFBS_ERR_STATE when nothing has been collected, when option "record_sites" was
 * off for that run, or when the run was a full scan ("delta" = 0, "record_matches" or the audit).  Pointers stay valid as those of
 * tfbs_rows do. */
int tfbs_get_record_sites(tfbs_ctx* ctx, tfbs_record_sites* out);

/* Matches of the last run when "record_matches" was on (call after tfbs_collect). */
int tfbs_get_matches(tfbs_ctx* ctx, tfbs_matches* out);

/* Audit of the block most recently given to tfbs_submit_block / tfbs_upload_block (it is still resident): scores it twice with
 * every distinct haplotype scanned in full, once with the thresholds lowered by one, and returns the windows that only the lowered
 * run reports (score == min_score) together with the per-haplotype flags.  Afterwards the context holds the results of a normal
 * run of the block (tfbs_collect works); options are left as they were.  Pointers stay valid until the next run. */
int tfbs_audit_block(tfbs_ctx* ctx, tfbs_audit* out);

/* Device-resident path for benchmarking: upload once, run the device pipeline on the
 * resident block any number of times.  tfbs_run_resident returns after the device work of
 * this run has been enqueued (two runs may be in flight, like tfbs_submit_block); tfbs_collect then fetches rows. */
int tfbs_upload_block(tfbs_ctx* ctx, const tfbs_block* block);
int tfbs_run_resident(tfbs_ctx* ctx);

int tfbs_get_stats(const tfbs_ctx* ctx, tfbs_stats* out);

/* Where the fan-out keeps its per-group count vectors (option "fan_vector").  *smem_groups: how many groups (distinct haplotypes of
 * a region, the reference haplotype included) a count vector in shared memory holds on this context's device; a block whose count
 * vector needs more capacity runs the fan-out with its vectors in device memory.  For the most recent run of the default path
 * (zeros before the first one, after a full scan, and for a block without keys): *groups_cap = the capacity of its count vector,
 * *ctas = the CTAs of the fan-out launch (in device memory: a fixed grid whose CTAs each own one count vector and walk the
 * region's units in turn, so a block with more regions than CTAs reuses every vector), *in_device_memory = 1 when the vectors were
 * in device memory, 0 when in shared memory. */
int tfbs_fanout_info(const tfbs_ctx* ctx, uint32_t* smem_groups, uint32_t* groups_cap, uint32_t* ctas, uint32_t* in_device_memory);

/* Page-lock / unlock caller buffers (cudaHostRegister) so that tfbs_submit_block copies them at full PCIe speed.
 * Optional: pageable buffers work, only slower. */
int tfbs_host_register(void* ptr, size_t bytes);
int tfbs_host_unregister(void* ptr);

/* The kernel stream (cudaStream_t) of the context's first lane: the pipelines of its blocks run on it, except, with option
 * "dual_stream", those of every other block of the default scoring mode, which run on the second lane's own kernel stream. */
void* tfbs_stream(const tfbs_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* TFBS_H */
