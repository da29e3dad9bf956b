// k2_types.cuh -- K2: pattern tables, count rows, match buffer, scan geometry
// Part of the sm_100a kernels of the find-tfbs hot path; included through kernels.cuh (see the map there).
#pragma once
#include "k1_build.cuh"

namespace tfbs {

// ------------------------------------------------------------------------------------------------
// K2: PWM scan
// ------------------------------------------------------------------------------------------------

struct DevPatterns {
    const u64* table;
    const ChunkDesc* chunks;
    const RunDesc* runs;
    const int* trip_pat;
    const u32* pat_len;
    const u32* pat_pid_index;
    const int* pat_w;  // [n_patterns][kMaxPatternLen][4] weights (option "sites": the rare path scores the windows it keeps)
    u32 n_chunks;
    u32 n_pid;       // distinct pattern ids
    u32 n_patterns;
    u32 max_len;
    u32 sum_len;
    u64 sum_len_sq;
};

struct DevCounts {
    u32* C;               // counts, [region][group][pid][inner]
    const u64* cbase;     // per region (block-wide), offset into C relative to cbase0
    u64 cbase0;
};

struct DevMatches {
    u32 enabled;
    u32 cap;
    u32* region;
    u32* pattern_index;
    u32* group;
    i64* start;
};

#ifndef TFBS_SCAN_WARPS
#define TFBS_SCAN_WARPS 24
#endif
#ifndef TFBS_SCAN_UNROLL
#define TFBS_SCAN_UNROLL 1   /* measured on B200: 1 -> 0.835 of the roof, 2 -> 0.775, 4 -> 0.61 (instruction cache) */
#endif
constexpr int SCAN_UNROLL = TFBS_SCAN_UNROLL;
constexpr int SCAN_WARPS = TFBS_SCAN_WARPS;          // warps per CTA; one CTA per SM shares one copy of the tables
constexpr int SCAN_CTA = SCAN_WARPS * 32;
#ifndef TFBS_TILE_POS
#define TFBS_TILE_POS 1024   /* multiple of 64; 2048 still fits next to 96 KB of tables (24 warps x 4.8 KB) */
#endif
#ifndef TFBS_MAX_PIECES
#define TFBS_MAX_PIECES 16
#endif
constexpr int TILE_POS = TFBS_TILE_POS;              // window starts staged per pass (per warp)
constexpr int PLANE_BYTES = TILE_POS / 2 + 32;       // pair codes of even / odd starts (+ halo)
constexpr int RAW_UNITS = TILE_POS / 32 + 3;
constexpr int MAX_RUNS = 16;
constexpr int MAX_PIECES = TFBS_MAX_PIECES;          // items (or tiles of a long item) scanned together by one warp
#ifndef TFBS_MERGE_GAP
#define TFBS_MERGE_GAP 0   /* measured on B200 (configs[1]): 0 -> 8.02 ms/step, 8 -> 8.26, 24 -> 9.05, 64 -> 12.5: short items are shared more */
#endif
// (Two variants of the per-iteration bookkeeping -- resuming the piece search, reading the pair codes as aligned words -- were timed
// on the B200 at the start of round 2: within 1.5 % of this code on both workloads, removed.)
#ifndef TFBS_PER_GRAB
#define TFBS_PER_GRAB 8
#endif
constexpr int SCAN_PER_GRAB = TFBS_PER_GRAB;         // list entries a warp takes per trip to the work counter under delta scoring
constexpr int MERGE_GAP = TFBS_MERGE_GAP;            // touched ranges closer than this are scored as one item (overlapping ones always are)

// Private to one warp: a warp owns the pieces of a round, so the scan needs no CTA-wide barrier.
struct __align__(16) WarpShared {
    u64 raw_pk[RAW_UNITS];
    u32 raw_nm[RAW_UNITS];
    u8 plane[2][PLANE_BYTES];
    // pieces of this round: window starts [p0, p0 + n) of item piece_item, staged at plane position pbase; vstart = starts before
    u32 piece_p0[MAX_PIECES], piece_vstart[MAX_PIECES + 1], piece_pbase[MAX_PIECES], piece_item[MAX_PIECES];
    u32 n_pieces, pad[3];
};

template <int FIELDS>
struct HitMask;
template <>
struct HitMask<3> { static constexpr u64 value = (1ULL << 20) | (1ULL << 41) | (1ULL << 62); };
template <>
struct HitMask<2> { static constexpr u64 value = (1ULL << 31) | (1ULL << 63); };

// Everything the rare path needs, passed by pointer (the structs are __grid_constant__ kernel parameters).
struct DevConfigs;
struct DevStatus;
struct ScanEnv {
    const DevConfigs* cf;   // configuration path (virtual sequences) or NULL
    const DevBlock* b;
    const DevSeqs* sq;
    const DevPatterns* pt;
    const DevCounts* ct;
    const DevMatches* mt;
    const DevRefHits* rh;
    DevStatus* st;
};

// One per CTA: the runs of the chunk and the bounds of the work list (read once per trip to the work counter).
struct __align__(16) CtaShared {
    RunDesc runs[MAX_RUNS];
    u32 n_runs;
    u32 per_grab;
    u64 n_list;
};

}  // namespace tfbs
