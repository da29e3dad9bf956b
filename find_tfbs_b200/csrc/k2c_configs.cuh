// k2c_configs.cuh -- K2, configuration path: what is scored under delta scoring, per (cluster of records, carried subset)
// Part of the sm_100a kernels of the find-tfbs hot path; included through kernels.cuh (see the map there).
//
// The reference scores every distinct haplotype of a region in full (main.rs:101-147).  Scores are integer sums and a hit is
// decided window by window, so the hits of a patched haplotype are the hits of the region's reference haplotype, minus those whose
// window touches a carried record, plus the hits of the windows that touch one.  Records further apart than the longest pattern
// never share a window: the in-window records of a region fall into CLUSTERS (a record joins the cluster of its predecessor unless
// at least Lmax - 1 untouched reference bases lie between them), and a haplotype is, cluster by cluster, one CONFIGURATION = the
// ordered list of the cluster's records it carries.  A configuration is scored once, as a virtual haplotype that carries nothing
// else, whatever number of haplotypes share it; k3_fanout.cuh adds the configurations' count differences up per distinct haplotype.
// patch_haplotype's truncation exit (haplotype.rs:144-149) drops everything behind it: a configuration that truncates loses every
// later reference hit, and the later configurations of such a haplotype are not applied.
#pragma once
#include "k2_worklist.cuh"

namespace tfbs {

// The sizes that only the device learns, each with a capacity the host chose (Caps, DevPlan::n / need).
struct Cap {
    enum : int {
        seq,        // distinct haplotypes (sequences)
        d,          // their in-window diff-list entries
        cfg,        // configurations
        vd,         // diff-list entries of the virtual sequences
        items,      // work-list items
        units,      // units of 32 packed bases
        dwords,     // words of the difference matrices
        rows,       // rows
        rowwords,   // packed row words
        capr,       // reference hits kept per region
        groups,     // groups a fan-out count vector holds
        terms,      // option "attribution": non-zero (row, configuration) differences (k3_attribution.cuh)
        sites_raw,  // options "sites" / "record_sites": raw sites, before gained / lost pairs cancel (k3_sites.cuh)
        sites,      // option "sites": the configurations' sites after the cancellation
        rsites,     // option "record_sites": the records' sites after the cancellation
        N
    };
};

// Sizes that are decided on the device.  Every stage is launched for a capacity the host chose; a gate kernel between two stages
// publishes the real count (clamped to the capacity), records the need and raises `abort` when the capacity was too small: the host
// then repeats the run with more scratch.  No stage ever comes back to the host.
struct DevPlan {
    u64 n[Cap::N];     // the counts, clamped to their capacity (none for capr and groups)
    u64 need[Cap::N];  // what the run needed, 0 where an earlier overflow left it unknown
    u64 n_vseq;        // virtual sequences: the reference haplotypes, the configurations, the records alone
    u64 n_members;     // entries of the configurations' member lists
    u64 n_sid;         // configurations + records alone: the virtual sequences behind the references, the ids the sites are ranked by
    u32 abort, cfg_collision;
    u64 unused;          // the need of the gates whose count is bounded by an earlier capacity (n_vseq, n_members)
    u64 rowwords_alloc;  // packed row words handed out by the fan-out (an atomic cursor)
    u64 fan_keys;        // keys the fan-out built a count vector for
    u64 fan_dbg[5];      // -DTFBS_FAN_STATS: pairs, member updates, groups with a non-zero difference, samples with one, keys of the dense pass
    u64 site_alloc;      // options "sites" / "record_sites": raw sites handed out by the rare path and k_cfg_lost (an atomic cursor)
};

// A count becomes known: total (+ add) against the capacity its consumers were launched for.  Behind an earlier overflow nothing
// is trustworthy: the count reads 0 (the later stages find nothing to do) and the need stays unknown.
__global__ void k_gate(const u64* total, u64 add, u64 cap, u64* n_out, u64* need_out, u32* abort_flag) {
    if (*abort_flag) { *need_out = 0; *n_out = 0; return; }
    const u64 need = *total + add;
    *need_out = need;
    if (need > cap) *abort_flag = 1;
    *n_out = need > cap ? cap : need;
}
// The same for the total of an exclusive scan over a device-side count: it sits behind the last scanned element.
__global__ void k_gate_at(const u64* offsets, const u64* n_ptr, u64 cap, u64* n_out, u64* need_out, u32* abort_flag) {
    if (*abort_flag) { *need_out = 0; *n_out = 0; return; }
    const u64 need = offsets[*n_ptr];
    *need_out = need;
    if (need > cap) *abort_flag = 1;
    *n_out = need > cap ? cap : need;
}

__global__ void k_zero_words(u32* p, const u64* n_ptr, u64 cap) {
    u64 n = *n_ptr < cap ? *n_ptr : cap;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) p[i] = 0;
}

// Options "sites" / "record_sites": a hit a configuration or a record alone gains (+1, rare path, mode 2) or a reference hit it loses
// (-1, k_cfg_lost), before equal (pattern, start, score) pairs cancel (k3_sites.cuh).
struct RawSite {
    u32 cfg;     // virtual configuration index (cfgbase[r] + column), or n_cfg + v for record v; the output id once k_site_scatter has grouped them
    u32 pat;     // pattern index
    int start;   // window start relative to region_start (pattern.rs:156)
    int score;   // exact window score
    int change;  // +1 gained, -1 lost
};

struct DevConfigs {
    u32 max_len;           // longest pattern (main.rs:404)
    u32 n_pid;
    // per record of the block
    u32* var_cluster;      // [n_var] cluster of an in-window record inside its region, 0xffffffff for the others
    u32* var_sorted;       // [n_var] scratch: the in-window records of a region by position
    // per region
    u32* ncfg;             // [R] configurations
    u64* cfgbase;          // [R+1] first configuration of the region
    u32* dwords;           // [R] ncfg * keys of the region
    u64* dbase;            // [R+1] first word of the region's difference matrix
    const u64* kbase;      // [R+1] first key of the region, keys = (pid, inner)
    // per entry e of the haplotypes' diff lists: runs of consecutive diffs of one cluster, described at their first entry
    u32* run_len;          // 0 = not the first entry of a live run
    u64* run_key;
    u32* run_rep;          // representative: the smallest e whose run holds the same records
    u32* run_cfg;          // at representatives: index of the configuration inside its region
    // per configuration
    u32* cfg_src;          // dlist index of the representative run
    int* cfg_net;          // hits gained minus reference hits lost
    u32* mcount;           // haplotype groups that carry it and are alive there
    u64* moff;             // [n_cfg+1]
    u32* mfill;
    u32* members;          // group numbers inside the region
    // counts
    u32* D;                // [region][key][configuration of the region]: difference to the reference haplotype's count (wrapping u32)
    u32* C0;               // [key] counts of the region's reference haplotype
    DevPlan* plan;
    // options "sites" / "record_sites" (site_raw NULL when both are off)
    RawSite* site_raw;     // [site_cap] in no particular order, behind plan->site_alloc
    u64 site_cap;
    u32* ref_pat;          // parallel to DevRefHits::buf: pattern index and score of each reference hit
    int* ref_score;
    u32 cfg_sites;         // option "sites": the configurations keep their sites too (with "record_sites" alone only the records do)
    u8* rec_flags;         // option "record_sites": [n_var] TFBS_REC_* of every record (k_cfg_walk)
};

__device__ __forceinline__ void put_site(const DevConfigs& cf, u32 c, u32 pat, int start, int score, int change) {
    const u64 k = atomicAdd(&cf.plan->site_alloc, 1ULL);
    if (k < cf.site_cap) cf.site_raw[k] = RawSite{c, pat, start, score, change};
}

// One CTA per region: the in-window records by position, cut into clusters.
__global__ void k_cluster(DevBlock b, DevConfigs cf) {
    const u32 r = blockIdx.x;
    const u32 v0 = b.var_off[r], v1 = b.var_off[r + 1];
    __shared__ u32 s_n;
    if (threadIdx.x == 0) s_n = 0;
    __syncthreads();
    for (u32 v = v0 + threadIdx.x; v < v1; v += blockDim.x) {
        cf.var_cluster[v] = 0xffffffffu;
        if (!b.var_inwin[v]) continue;
        const i64 p = b.variants[v].pos;
        u32 rank = 0;
        for (u32 u = v0; u < v1; ++u)
            if (b.var_inwin[u]) {
                const i64 pu = b.variants[u].pos;
                rank += (pu < p || (pu == p && u < v)) ? 1u : 0u;
            }
        cf.var_sorted[v0 + rank] = v;
        atomicAdd(&s_n, 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const i64 gap = cf.max_len ? (i64)cf.max_len : 1;
        i64 reach = 0;
        u32 cl = 0;
        for (u32 k = 0; k < s_n; ++k) {
            const u32 v = cf.var_sorted[v0 + k];
            const tfbs_variant x = b.variants[v];
            if (k > 0 && x.pos >= reach + gap) ++cl;  // at least Lmax - 1 untouched reference bases since the last consumed one
            cf.var_cluster[v] = cl;
            const i64 last = x.pos + (i64)x.ref_len - 1;
            if (k == 0 || last > reach) reach = last;
        }
    }
}

__device__ __forceinline__ u64 run_hash(u64 h, u32 v) { return mix64(h ^ ((u64)v * 0x9e3779b97f4a7c15ULL)) + 0x632be59bd9b4e019ULL; }

// Thread per distinct haplotype: its consumed diffs, cut where the cluster changes.  The smallest entry index with the same key
// becomes the representative of the configuration.
__global__ void k_cfg_runs(DevBlock b, DevSeqs sq, DevConfigs cf, u64 d_cap, u64 seed, u64* keys, u32* vals, u32 mask) {
    if (cf.plan->abort) return;
    const u32 q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= seq_count(sq)) return;
    const u64 doff = sq.seq_doff[q];
    const u32 nd = sq.seq_nd[q];
    if (doff + nd > d_cap) return;
    const u32* dl = sq.dlist + doff;
    for (u32 k = 0; k < nd; ++k) cf.run_len[doff + k] = 0;
    if (sq.seq_flags[q] & 2) return;  // overwritten in the sequence-keyed map: counted with the reference haplotype
    const u32 ntake = sq.seq_ntake[q] < nd ? sq.seq_ntake[q] : nd;
    const u32 r = sq.seq_region[q];
    for (u32 k = 0; k < ntake;) {
        const u32 c = cf.var_cluster[dl[k]];
        u64 h = mix64(seed ^ ((u64)(r + 1) << 32) ^ c);
        u32 j = k;
        while (j < ntake && cf.var_cluster[dl[j]] == c) { h = run_hash(h, dl[j]); ++j; }
        const u64 key = h | 1ULL;
        cf.run_len[doff + k] = j - k;
        cf.run_key[doff + k] = key;
        atomicMin(&vals[table_find_or_insert(keys, mask, key)], (u32)(doff + k));
        k = j;
    }
}

// Thread per distinct haplotype: every run learns its representative (verified record by record: a hash collision makes the host
// repeat the run with another seed) and the representative numbers the configuration inside its region.
__global__ void k_cfg_resolve(DevSeqs sq, DevConfigs cf, u64 d_cap, const u64* keys, const u32* vals, u32 mask) {
    if (cf.plan->abort) return;
    const u32 q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= seq_count(sq)) return;
    const u64 doff = sq.seq_doff[q];
    const u32 nd = sq.seq_nd[q];
    if (doff + nd > d_cap) return;
    const u32 r = sq.seq_region[q];
    for (u32 k = 0; k < nd; ++k) {
        const u64 e = doff + k;
        const u32 n = cf.run_len[e];
        if (!n) continue;
        const u32 rep = vals[table_find(keys, mask, cf.run_key[e])];
        cf.run_rep[e] = rep;
        if (rep == (u32)e) {
            cf.run_cfg[e] = atomicAdd(&cf.ncfg[r], 1u);
        } else {
            bool same = cf.run_len[rep] == n;
            for (u32 x = 0; same && x < n; ++x) same = sq.dlist[rep + x] == sq.dlist[e + x];
            if (!same) cf.plan->cfg_collision = 1;
        }
    }
}

__global__ void k_region_sizes(DevBlock b, DevConfigs cf) {
    const u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= b.R) return;
    const u64 nkeys = (u64)cf.n_pid * (b.inner_off[r + 1] - b.inner_off[r]);
    const u64 w = (u64)cf.ncfg[r] * nkeys;
    cf.dwords[r] = w > 0xffffffffULL ? 0xffffffffu : (u32)w;
    if (w > 0xffffffffULL) cf.plan->abort = 1;  // a single region with more than 2^32 (configuration, key) pairs: not representable
}

// Virtual sequences: q < R is the reference haplotype of region q, R + cfgbase[r] + c configuration c of region r, and (option
// "record_sites", n_rec = the block's records) R + n_cfg + v record v alone: its diff list is [v], empty outside its region's window.
__global__ void k_vseq_init(DevBlock b, DevConfigs cf, DevSeqs vq, u32 n_rec) {
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t == 0) cf.plan->n_sid = cf.plan->n[Cap::cfg] + n_rec;
    if (t < b.R && t < vq.n_seq) {
        vq.seq_region[t] = t;
        vq.seq_leader[t] = 0xffffffffu;
        vq.seq_nd[t] = 0;
    }
    if (t >= n_rec || cf.plan->abort) return;
    const u64 u = (u64)vq.n_ref + cf.plan->n[Cap::cfg] + t;
    if (u >= vq.n_seq) return;
    u32 lo = 0, hi = b.R;  // the region of record t: the last r with var_off[r] <= t
    while (hi - lo > 1) {
        const u32 mid = (lo + hi) / 2;
        if (b.var_off[mid] <= t) lo = mid; else hi = mid;
    }
    vq.seq_region[u] = lo;
    vq.seq_leader[u] = 0xffffffffu;
    vq.seq_nd[u] = b.var_inwin[t] ? 1u : 0u;
}
__global__ void k_cfg_fill(DevSeqs sq, DevConfigs cf, DevSeqs vq, u64 d_cap) {
    if (cf.plan->abort) return;
    const u32 q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= seq_count(sq)) return;
    const u64 doff = sq.seq_doff[q];
    const u32 nd = sq.seq_nd[q];
    if (doff + nd > d_cap) return;
    const u32 r = sq.seq_region[q];
    for (u32 k = 0; k < nd; ++k) {
        const u64 e = doff + k;
        if (!cf.run_len[e] || cf.run_rep[e] != (u32)e) continue;
        const u64 c = cf.cfgbase[r] + cf.run_cfg[e];
        const u64 u = (u64)vq.n_ref + c;
        if (u >= vq.n_seq) continue;
        vq.seq_region[u] = r;
        vq.seq_leader[u] = q;  // the haplotype group the representative run belongs to (informational)
        vq.seq_nd[u] = cf.run_len[e];
        cf.cfg_src[c] = (u32)e;
        cf.cfg_net[c] = 0;
    }
}

// Thread per virtual sequence: the configuration's records walked like patch_haplotype would walk a haplotype that carries only them.
// A record alone that lies outside the window or meets one of patch_haplotype's panics gets its flag and length 0 (no windows): only
// a haplotype's own walk (k_walk) fails the block.
__global__ void k_cfg_walk(DevBlock b, DevSeqs sq, DevConfigs cf, DevSeqs vq, u64 vd_cap) {
    if (cf.plan->abort) return;
    const u32 u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= seq_count(vq)) return;
    const u64 doff = vq.seq_doff[u];
    const u32 nd = vq.seq_nd[u];
    if (doff + nd > vd_cap) return;
    u32* dl = vq.dlist + doff;
    const u64 c = (u64)u - vq.n_ref, n_cfg = cf.plan->n[Cap::cfg];
    const bool rec = u >= vq.n_ref && c >= n_cfg;
    if (rec) {
        if (nd) dl[0] = (u32)(c - n_cfg);
    } else if (u >= vq.n_ref) {
        const u32* src = sq.dlist + cf.cfg_src[c];
        for (u32 k = 0; k < nd; ++k) dl[k] = src[k];
    }
    Seg* sg = vq.segs + 2 * doff + 2 * (u64)u;
    const WalkOut w = walk_diffs(b, vq.seq_region[u], dl, nd, sg, nullptr, 0);
    vq.seq_nseg[u] = w.ns;
    vq.seq_len[u] = w.len;
    vq.seq_flags[u] = w.trunc ? 1 : 0;
    vq.seq_ntake[u] = w.ntake;
    if (rec) {
        const u8 f = !nd ? (u8)TFBS_REC_OUTSIDE
                   : w.err == DEV_REF_MISMATCH ? (u8)TFBS_REC_REF_MISMATCH : w.err == DEV_MISSING_CASE ? (u8)TFBS_REC_MISSING_CASE : (u8)0;
        cf.rec_flags[c - n_cfg] = f;
        if (f) vq.seq_len[u] = 0;
    }
}

// Work list over the virtual sequences: the reference haplotype of a region in full, a configuration only at the window starts
// that touch one of its ALT segments ([a - Lmax + 1, e - 1] for a segment [a, e)): every other window lies inside one
// reference-copy segment and has the bases and positions of the reference window there.
constexpr u32 REF_PIECE = 128;
template <bool FILL>
__global__ void k_vitems(DevSeqs vq, u32 max_len, const u32* abort_flag) {
    if (*abort_flag) return;
    const u32 q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= seq_count(vq)) return;
    const u32 len = vq.seq_len[q];
    u32 n = 0;
    const u64 base = FILL ? vq.item_off[q] : 0;
    auto put = [&](u32 a, u32 z) {
        if (FILL && base + n < vq.n_items_cap) vq.items[base + n] = ScanItem{q, a, z, (u32)(base + n)};
        ++n;
    };
    if (len == 0) {
        n = 0;
    } else if (q < vq.n_ref) {
        // the reference haplotype in pieces of REF_PIECE starts: a trip to the scan's work counter then costs about the same
        // whether it draws pieces of a reference haplotype or short items of configurations
        for (u32 a = 0; a < len; a += REF_PIECE) put(a, (a + REF_PIECE < len ? a + REF_PIECE : len) - 1);
    } else {
        const Seg* sg = vq.segs + 2 * vq.seq_doff[q] + 2 * (u64)q;
        const u32 ns = vq.seq_nseg[q];
        bool open = false;
        u32 a = 0, z = 0;
        auto add = [&](long long lo, long long hi) {  // window starts [lo, hi], ascending lo
            if (lo < 0) lo = 0;
            if (hi > (long long)len - 1) hi = (long long)len - 1;
            if (hi < lo) return;
            if (open && (u32)lo <= z + MERGE_GAP) { if ((u32)hi > z) z = (u32)hi; return; }
            if (open) put(a, z);
            a = (u32)lo; z = (u32)hi; open = true;
        };
        for (u32 s = 0; s < ns; ++s) {
            const long long bb = sg[s].out_start, e = sg[s + 1].out_start;
            if (sg[s].kind == 1) add(bb - (long long)max_len + 1, e - 1);
            else if (s > 0 && sg[s - 1].kind == 0) add(bb - (long long)max_len + 1, bb - 1);
        }
        if (open) put(a, z);
    }
    if (!FILL) vq.seq_nitems[q] = n;
}

// Every item of the virtual work list is scored: the list is the identity, an entry needs the packed bases [p0 & ~31, p1 + 64].
__global__ void k_vitem_units(DevSeqs vq, const u64* n_items_ptr, u32* list) {
    const u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= *n_items_ptr || (vq.abort && *vq.abort)) return;
    list[w] = (u32)w;
    const ScanItem it = vq.items[w];
    vq.ent_units[w] = ((it.p1 + 64) >> 5) - (it.p0 >> 5) + 1;
}

// 8 lanes per configuration: the hits of the region's reference haplotype that the configuration does not inherit (the window is
// not inside ONE of its reference-copy segments; behind a truncation nothing is) are taken out of its column of the difference matrix.
// A record alone (option "record_sites") only lists them as lost sites; one without windows (a flag, k_cfg_walk) has none.
__global__ void k_cfg_lost(DevBlock b, DevSeqs vq, DevConfigs cf, DevRefHits rh) {
    if (cf.plan->abort) return;
    constexpr u32 GS = 8;
    const u32 u = vq.n_ref + (blockIdx.x * blockDim.x + threadIdx.x) / GS;
    const u32 lane = threadIdx.x % GS;
    if (u >= seq_count(vq)) return;
    const bool rec = (u64)u - vq.n_ref >= cf.plan->n[Cap::cfg];
    if (rec && vq.seq_len[u] == 0) return;
    const u32 r = vq.seq_region[u];
    const u32 nh = min(rh.cnt[r - rh.r0], rh.capr);
    const u32 nk = b.inner_off[r + 1] - b.inner_off[r];
    const tfbs_inner_region* inner = b.inner + b.inner_off[r];
    const i64 rs = b.region_start[r];
    const u64 c = (u64)u - vq.n_ref;
    const u32 ncfg = cf.ncfg[r];
    u32* col = cf.D + cf.dbase[r] + (c - cf.cfgbase[r]);
    const Seg* sg = vq.segs + 2 * vq.seq_doff[u] + 2 * (u64)u;
    const u32 ns = vq.seq_nseg[u];
    const RefHit* hits = rh.buf + (u64)(r - rh.r0) * rh.capr;
    int lost = 0;
    for (u32 j = lane; j < nh; j += GS) {
        const RefHit h = hits[j];
        bool inside = false;
        for (u32 s = 0; s < ns && !inside; ++s)
            inside = sg[s].kind == 0 && sg[s].relpos <= h.relpos &&
                     (i64)h.relpos + h.len <= (i64)sg[s].relpos + (i64)(sg[s + 1].out_start - sg[s].out_start);
        if (inside) continue;
        ++lost;
        if (cf.site_raw && (rec || cf.cfg_sites)) {
            const u64 x = (u64)(r - rh.r0) * rh.capr + j;
            put_site(cf, (u32)c, cf.ref_pat[x], h.relpos, cf.ref_score[x], -1);
        }
        if (rec) continue;
        const i64 hs = h.relpos, he = hs + h.len - 1;
        for (u32 k = 0; k < nk; ++k) {
            i64 is = inner[k].start - rs, ie = inner[k].end - rs;
            if ((hs >= is && hs <= ie) || (he >= is && he <= ie)) atomicSub(&col[((u64)h.pid * nk + k) * ncfg], inner[k].multiplicity);
        }
    }
    if (lost && !rec) atomicSub(&cf.cfg_net[c], lost);
}

__global__ void k_refhit_need(DevRefHits rh, u32 nr, DevPlan* plan) {
    const u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nr) return;
    const u32 n = rh.cnt[r];
    if (n > rh.capr) plan->abort = 1;
    atomicMax(&plan->need[Cap::capr], (u64)n);
}

// Members of the configurations (thread per distinct haplotype, twice: count, then fill).  The fill pass also adds up the work
// counters of the scanned haplotypes: hits (the reference haplotype's hits plus the net hits of the live configurations), executed
// cells (pattern.rs:147-150 on the haplotype's length) and their number.
template <bool FILL>
__global__ void k_members(DevSeqs sq, DevConfigs cf, DevRefHits rh, const u32* ref_used, u64 d_cap, DevPatterns pt, DevStatus* st) {
    __shared__ unsigned long long s_hits, s_cells;
    __shared__ u32 s_scanned;
    if (FILL) {
        if (threadIdx.x == 0) { s_hits = 0; s_cells = 0; s_scanned = 0; }
        __syncthreads();
    }
    const u32 q = blockIdx.x * blockDim.x + threadIdx.x;
    long long hits = 0;
    u64 cells = 0;
    u32 scanned = 0;
    if (!cf.plan->abort && q < seq_count(sq)) {
        const u64 doff = sq.seq_doff[q];
        const u32 nd = sq.seq_nd[q];
        const u32 r = sq.seq_region[q];
        const u32 g = seq_group(sq, q);
        if (doff + nd <= d_cap) {
            if (FILL && seq_is_scanned(sq, q, ref_used)) {
                hits = (long long)min(rh.cnt[r - rh.r0], rh.capr);
                scanned = 1;
                cells = cells_of_length(sq.seq_len[q], pt.max_len, pt.sum_len, pt.sum_len_sq, pt.n_patterns, pt.pat_len);
            }
            for (u32 k = 0; k < nd; ++k) {
                const u64 e = doff + k;
                if (!cf.run_len[e]) continue;
                const u64 c = cf.cfgbase[r] + cf.run_cfg[cf.run_rep[e]];
                if (!FILL) atomicAdd(&cf.mcount[c], 1u);
                else {
                    const u64 slot = cf.moff[c] + atomicAdd(&cf.mfill[c], 1u);
                    if (slot < d_cap) cf.members[slot] = g;
                    hits += cf.cfg_net[c];
                }
            }
        }
    }
    if (FILL) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            hits += __shfl_xor_sync(0xffffffffu, hits, o);
            cells += __shfl_xor_sync(0xffffffffu, cells, o);
            scanned += __shfl_xor_sync(0xffffffffu, scanned, o);
        }
        if ((threadIdx.x & 31) == 0) {
            if (hits) atomicAdd(&s_hits, (unsigned long long)hits);
            if (cells) atomicAdd(&s_cells, (unsigned long long)cells);
            if (scanned) atomicAdd(&s_scanned, scanned);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            if (s_hits) atomicAdd(&st->n_hits, s_hits);
            if (s_cells) atomicAdd(&st->executed_cells, s_cells);
            if (s_scanned) atomicAdd(&st->n_scanned, (u64)s_scanned);
        }
    }
}

}  // namespace tfbs
