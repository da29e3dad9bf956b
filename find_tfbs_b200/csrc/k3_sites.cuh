// k3_sites.cuh -- K3, configuration path, options "sites" and "record_sites": the binding sites behind each attribution term, and
// those of every record of the block alone
// Part of the sm_100a kernels of the find-tfbs hot path; included through kernels.cuh (see the map there).
//
// A configuration's sites are two multiset differences of (pattern, start, score) hit triples: gained = A - R and lost = R - A, where
// A holds the hits of the region's window patched with the configuration's records alone and R those of the unpatched window.  Every
// window a configuration inherits has the same bases and start in both, so they are the rare path's mode-2 hits (+1) against the
// reference hits k_cfg_lost takes out (-1), after equal triples cancel in pairs (a window of identical bases that touches an ALT
// segment, e.g. one that ends on a deletion's anchor base, is in both lists).  Those raw sites arrive in no particular order
// (RawSite, DevConfigs::site_raw); the launches here run right behind the attribution kernels and lay them out per output id.  A record
// alone (option "record_sites") is one more virtual configuration with a one-entry diff list; its id n_cfg + v follows the
// configurations' output ids, so one ranking serves both:
//   1. count per output id (site_oid, written by k_att_configs<false>; a record's id is its own), scan, scatter: the sites grouped by id;
//   2. a CTA per configuration ranks its sites by (pattern, start, score, change), tile by tile through shared memory, into the sorted
//      order, and flags the survivors: of n_lost -1 and n_gained +1 entries of one triple, the first n_lost - m and the last
//      n_gained - m stay (m = min(n_lost, n_gained));
//   3. a scan of the flags numbers the survivors block-wide (configurations are consecutive in output-id order, the records behind
//      them), a gate checks the two result capacities, and one pass writes them and the per-configuration and per-record offsets.
// Nothing depends on hash seeds, atomics or the lane: the output is a function of the multiset of raw sites.
#pragma once
#include "k3_attribution.cuh"

namespace tfbs {

constexpr int SITE_THREADS = 128;

struct DevSites {
    // scratch (shared by consecutive blocks)
    RawSite* raw;       // [Cap::sites_raw] the raw sites (DevConfigs::site_raw); after the scatter, the sorted order
    RawSite* bucket;    // [Cap::sites_raw] grouped by output id
    u32* keep;          // [Cap::sites_raw] 1 at a surviving site of the sorted order
    u64* kpos;          // [Cap::sites_raw + 1] exclusive scan of keep: the survivor's output index
    const u32* oid;     // [cfg] output id of each virtual configuration (DevAttr::site_oid)
    u32* cnt;           // [cfg + records] raw sites per output id
    u64* boff;          // [cfg + records + 1] exclusive scan of cnt
    const u64* n_cfg;   // DevPlan::n[Cap::cfg]: ids from n_cfg on are records
    // results (per slot): option "sites" (site_off NULL when off)
    u64* site_off;      // [cfg + 1]
    u32* pat;           // [sites]
    i64* start;
    int* score;
    signed char* change;
    const u32* cfg_region;  // DevAttr::cfg_region
    // results (per slot): option "record_sites" (rec_off NULL when off)
    u64* rec_off;       // [records + 1]
    u32* rec_pat;       // [record sites]
    i64* rec_start;
    int* rec_score;
    signed char* rec_change;
    const u32* vseq_region;  // DevSeqs::seq_region of the virtual sequences: id o >= n_cfg is the sequence n_ref + o
    u32 n_ref;
};

__device__ __forceinline__ u32 site_out_id(const DevSites& s, u32 c) { return c < *s.n_cfg ? s.oid[c] : c; }

__device__ __forceinline__ bool site_less(const RawSite& a, const RawSite& b) {
    if (a.pat != b.pat) return a.pat < b.pat;
    if (a.start != b.start) return a.start < b.start;
    if (a.score != b.score) return a.score < b.score;
    return a.change < b.change;
}

__global__ void k_site_count(DevSites s, const u64* n_raw_ptr, const u32* abort_flag) {
    if (*abort_flag) return;
    const u64 n = *n_raw_ptr;
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (u64)gridDim.x * blockDim.x) atomicAdd(&s.cnt[site_out_id(s, s.raw[k].cfg)], 1u);
}

// cnt is counted down again: it ends all zero.
__global__ void k_site_scatter(DevSites s, const u64* n_raw_ptr, const u32* abort_flag) {
    if (*abort_flag) return;
    const u64 n = *n_raw_ptr;
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (u64)gridDim.x * blockDim.x) {
        RawSite x = s.raw[k];
        x.cfg = site_out_id(s, x.cfg);
        s.bucket[s.boff[x.cfg] + atomicSub(&s.cnt[x.cfg], 1u) - 1] = x;
    }
}

// CTAs walk the output ids; every thread ranks one site of the configuration per pass against all of them (n^2 compares through
// shared-memory tiles: tens of sites usually, tens of thousands for an always-hit pattern under a long insertion).  A site's rank is
// the sites with a smaller key plus the equal ones before it; `eq` = its index among equal keys.
__global__ void __launch_bounds__(SITE_THREADS) k_site_rank(DevSites s, const u64* n_id_ptr, const u32* abort_flag) {
    __shared__ RawSite tile[SITE_THREADS];
    if (*abort_flag) return;
    const u64 n_id = *n_id_ptr;
    for (u64 o = blockIdx.x; o < n_id; o += gridDim.x) {
        const u64 b0 = s.boff[o], n = s.boff[o + 1] - b0;
        for (u64 i0 = 0; i0 < n; i0 += SITE_THREADS) {
            const u64 i = i0 + threadIdx.x;
            const RawSite mine = i < n ? s.bucket[b0 + i] : RawSite{};
            u64 less = 0, eq = 0, n_lost = 0, n_gained = 0;
            for (u64 t0 = 0; t0 < n; t0 += SITE_THREADS) {
                __syncthreads();
                if (t0 + threadIdx.x < n) tile[threadIdx.x] = s.bucket[b0 + t0 + threadIdx.x];
                __syncthreads();
                const u32 m = (u32)(n - t0 < (u64)SITE_THREADS ? n - t0 : (u64)SITE_THREADS);
                for (u32 k = 0; k < m; ++k) {
                    const RawSite y = tile[k];
                    const bool same = y.pat == mine.pat && y.start == mine.start && y.score == mine.score;
                    less += site_less(y, mine) ? 1u : 0u;
                    eq += (same && y.change == mine.change && t0 + k < i) ? 1u : 0u;
                    n_lost += (same && y.change < 0) ? 1u : 0u;
                    n_gained += (same && y.change > 0) ? 1u : 0u;
                }
            }
            if (i < n) {
                const u64 m = n_lost < n_gained ? n_lost : n_gained;
                const bool keep = mine.change < 0 ? eq < n_lost - m : eq >= m;
                s.raw[b0 + less + eq] = mine;
                s.keep[b0 + less + eq] = keep ? 1u : 0u;
            }
        }
        __syncthreads();
    }
}

// The survivors of the configurations and those of the records against their result capacities (as k_gate_at does for one count).
__global__ void k_site_gate(DevSites s, const u64* n_raw_ptr, u64 cap_cfg, u64 cap_rec, DevPlan* plan) {
    if (plan->abort) { plan->need[Cap::sites] = plan->n[Cap::sites] = plan->need[Cap::rsites] = plan->n[Cap::rsites] = 0; return; }
    const u64 all = s.kpos[*n_raw_ptr], in_cfg = s.kpos[s.boff[*s.n_cfg]];
    plan->need[Cap::sites] = in_cfg;
    plan->need[Cap::rsites] = all - in_cfg;
    if (in_cfg > cap_cfg || all - in_cfg > cap_rec) plan->abort = 1;
    plan->n[Cap::sites] = in_cfg > cap_cfg ? cap_cfg : in_cfg;
    plan->n[Cap::rsites] = all - in_cfg > cap_rec ? cap_rec : all - in_cfg;
}

// The survivors in sorted order behind their block-wide index (the records' behind those of the configurations), site_off[o] = the
// survivors of the configurations before o, rec_off[v] = those of the records before v.
__global__ void k_site_emit(DevBlock b, DevSites s, const u64* n_raw_ptr, const u64* n_id_ptr, const u32* abort_flag) {
    if (*abort_flag) return;
    const u64 n = *n_raw_ptr, n_id = *n_id_ptr, n_cfg = *s.n_cfg;
    const u64 cfg_end = s.kpos[s.boff[n_cfg]];
    const u64 end = n > n_id + 1 ? n : n_id + 1;
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < end; k += (u64)gridDim.x * blockDim.x) {
        if (s.site_off && k <= n_cfg) s.site_off[k] = s.kpos[s.boff[k]];
        if (s.rec_off && k >= n_cfg && k <= n_id) s.rec_off[k - n_cfg] = s.kpos[s.boff[k]] - cfg_end;
        if (k >= n || !s.keep[k]) continue;
        const RawSite x = s.raw[k];
        const u64 p = s.kpos[k];
        if (x.cfg < n_cfg) {
            s.pat[p] = x.pat;
            s.start[p] = b.region_start[s.cfg_region[x.cfg]] + x.start;
            s.score[p] = x.score;
            s.change[p] = (signed char)x.change;
        } else {
            const u64 q = p - cfg_end;
            s.rec_pat[q] = x.pat;
            s.rec_start[q] = b.region_start[s.vseq_region[(u64)s.n_ref + x.cfg]] + x.start;
            s.rec_score[q] = x.score;
            s.rec_change[q] = (signed char)x.change;
        }
    }
}

}  // namespace tfbs
