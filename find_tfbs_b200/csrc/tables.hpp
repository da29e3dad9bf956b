// tables.hpp -- host-side compilation of the pattern list into the shared-memory lookup tables
// the scan kernel reads.
//
// Reference semantics (Helkafen/find-tfbs): a window scores sum_c weights[c].acgtn[nuc(i+c)] with the N
// slot = 0 (src/types.rs:103-113, src/pattern.rs:119-129) and is a hit iff score > min_score
// (src/pattern.rs:151).  Scores are exact i32, so any regrouping of the sum is exact.
//
// Layout idea: two adjacent columns are folded into one 25-entry table indexed by the pair of bases
// (16 ACGT pairs first, the 9 pairs involving N after them), and the entries of up to three patterns
// are packed into one 64-bit word as biased non-negative fields.  One LDS.64 then advances three
// patterns by two columns.  Field f of a word holds (w[c][a]-m[c]) + (w[c+1][b]-m[c+1]) with
// m[c] = min(0, min_x w[c][x]); the first pair additionally holds BIAS = FLAG-1-(min_score - sum m), so
// that after the last pair bit FLAG of the field is set iff score > min_score.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/tfbs.h"

namespace tfbs {

constexpr int kPairEntries = 25;   // 16 ACGT pairs + 9 pairs with N
constexpr int kMaxGroups = 16;     // column pairs per pattern in the fast kernel => L <= 32
constexpr int kMaxPatternLen = 2 * kMaxGroups;

// entry index of the base pair (a, b), a and b in 0..4 (4 = N).
inline int pair_entry(int a, int b) {
    if (a < 4 && b < 4) return 4 * a + b;
    if (a == 4) return 16 + b;          // N? -> 16..20
    return 21 + a;                      // ?N with a in 0..3 -> 21..24
}

struct HostPattern {
    std::vector<int32_t> w;  // len x 4
    uint32_t len = 0;
    int32_t min_score = 0;
    uint16_t pattern_id = 0;
    uint8_t direction = 0;
    uint8_t kind = 0;
    uint32_t pid_index = 0;  // index into the sorted list of distinct pattern_ids
};

struct RunDesc {
    uint32_t groups;     // column pairs of every triple in this run
    uint32_t n_triples;
};

// One chunk = a set of pattern_ids whose tables are resident in shared memory together.
struct ChunkDesc {
    uint32_t tbl_off;     // first 64-bit word of the chunk in the table blob
    uint32_t tbl_words;
    uint32_t trip_off;    // first triple (index into trip_pat / 'fields' slots per triple)
    uint32_t n_triples;
    uint32_t run_off;
    uint32_t n_runs;
    uint32_t pid_lo;      // pid_index range [pid_lo, pid_lo + n_pid)
    uint32_t n_pid;
    uint32_t fields;      // 3 = three 21-bit fields per word, 2 = two 32-bit fields
    uint32_t reserved;
};

struct CompiledPatterns {
    std::vector<HostPattern> patterns;       // as given, PWM and Other
    std::vector<uint16_t> pid_list;          // distinct pattern_ids, ascending
    std::vector<uint64_t> table;             // all chunks
    std::vector<ChunkDesc> chunks;
    std::vector<RunDesc> runs;
    std::vector<int32_t> trip_pat;           // 3 slots per triple (unused slots -1): index into patterns
    std::vector<uint32_t> pat_len;           // per pattern
    std::vector<uint32_t> pat_pid_index;     // per pattern
    std::vector<int32_t> pat_w;              // per pattern kMaxPatternLen x 4 weights, zero behind its length (option "sites" scores hits)
    uint32_t max_len = 0;                    // max pattern_length over all patterns (main.rs:404)
    uint32_t sum_len = 0;                    // sum of L over PWM patterns
    uint64_t sum_len_sq = 0;                 // sum of L*(L-1)
    uint32_t max_chunk_bytes = 0;
    uint32_t fields = 3;                     // 3 x 21-bit or 2 x 32-bit fields per table word (all chunks alike)
};

// Returns TFBS_OK or an error code with *err filled in.  table_budget_bytes bounds one chunk's tables.
int compile_patterns(const tfbs_pattern* patterns, uint32_t n, uint32_t table_budget_bytes, int force_wide,
                     CompiledPatterns* out, std::string* err);

}  // namespace tfbs
