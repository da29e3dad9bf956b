// k2_scan.cuh -- K2: the PWM scan kernel and its rare path
// Part of the sm_100a kernels of the find-tfbs hot path; included through kernels.cuh (see the map there).
#pragma once
#include "k2_types.cuh"
#include "k2c_configs.cuh"

namespace tfbs {

// Option "sites": the exact score of a hit, from the pattern's weights and the packed bases of the list entry (N scores 0).  On the
// configuration path the work list is the identity (k_vitem_units), so the item is the entry, and its units hold the bases
// [p0 & ~31, p1 + 64]: a window [i, i + L) with p0 <= i <= p1 and L <= 32 lies inside.  Then the site is kept: a configuration's or a
// record's hit goes to the raw site list (+1), a hit of the reference haplotype is remembered next to its RefHit slot (k_cfg_lost takes
// the lost ones).
__device__ __forceinline__ void keep_site(const ScanEnv* env, u32 mode, u64 at, u32 entry, u32 pi, u32 i, u32 L, int hs) {
    const DevSeqs& sq = *env->sq;
    const DevConfigs& cf = *env->cf;
    const u64* pk = sq.pk + sq.ent_uoff[entry];
    const u32* nm = sq.nm + sq.ent_uoff[entry];
    const int* w = env->pt->pat_w + (u64)pi * (kMaxPatternLen * 4);
    const u32 base = sq.items[entry].p0 & ~31u;
    int score = 0;
    for (u32 k = 0; k < L; ++k) {
        const u32 x = i + k - base;
        if (!((nm[x >> 5] >> (x & 31)) & 1u)) score += w[4 * k + ((u32)(pk[x >> 5] >> (2 * (x & 31))) & 3u)];
    }
    if (mode == 2) {
        put_site(cf, (u32)at, pi, hs, score, 1);
    } else {
        cf.ref_pat[at] = pi;
        cf.ref_score[at] = score;
    }
}

// Rare path: a window scored above the threshold in at least one field.  SITES (a k_scan of its own, so that the registers and the
// stack of the scan without options "sites" and "record_sites" stay as they are): the sites are kept too (keep_site), and the virtual
// sequences behind the configurations are records alone, whose hits are sites only.
template <bool SITES>
__device__ __noinline__ u32 scan_on_hit(u64 hit, u32 t, u32 i, u32 item_index, ChunkDesc cd, const ScanEnv* env) {
    u32 counted = 0;  // hits of a full scan: the caller adds them to the statistics once per work grab
    const DevSeqs& sq = *env->sq;
    const DevBlock& b = *env->b;
    const DevPatterns& pt = *env->pt;
    DevStatus* st = env->st;
    const ScanItem item = sq.items[item_index];
    const u32 q = item.q;
    const u32 len = sq.seq_len[q];
    const u32 nseg = sq.seq_nseg[q];
    const Seg* sg = sq.segs + 2 * sq.seq_doff[q] + 2 * (u64)q;
    const u32 r = sq.seq_region[q];
    const u32 g = seq_group(sq, q);
    // 0 full scan: count every hit into the row of the haplotype's group; configuration path: 1 reference haplotype (count + remember
    // the hit), 2 configuration: count only windows that touch one of its records, into its column of the difference matrix
    const u32 mode = env->cf ? (g == 0 ? 1u : 2u) : 0u;
    const u32 nk = b.inner_off[r + 1] - b.inner_off[r];
    const tfbs_inner_region* inner = b.inner + b.inner_off[r];
    const i64 region_start = b.region_start[r];
    const int bits = cd.fields == 3 ? 21 : 32;
    for (u32 f = 0; f < cd.fields; ++f) {
        if (!((hit >> (bits * f + bits - 1)) & 1ULL)) continue;
        int pi = pt.trip_pat[(size_t)(cd.trip_off + t) * 3 + f];
        if (pi < 0) continue;
        u32 L = pt.pat_len[pi];
        if (i + L > len) continue;  // pattern.rs:147-149: only complete windows
        // pos of the first base of the window (pattern.rs:156)
        u32 s = seg_find(sg, nseg, i);
        Seg cur = sg[s];
        if (mode == 2 && cur.kind == 0 && i + L <= sg[s + 1].out_start) continue;  // untouched window: inherited from the reference
        i64 hs = (i64)cur.relpos + (cur.kind == 0 ? (i64)(i - cur.out_start) : 0);
        i64 he = hs + L - 1;
        u32 pl = pt.pat_pid_index[pi];
        u32* crow;
        u64 cstride = 1;
        if (mode == 2) {  // a configuration: its column of the region's difference matrix D[key][configuration]
            const DevConfigs& cf = *env->cf;
            const u64 c = (u64)q - sq.n_ref;
            if (SITES && c >= cf.plan->n[Cap::cfg]) {  // a record alone (option "record_sites"): nothing is counted
                keep_site(env, 2, c, item_index, (u32)pi, i, L, (int)hs);
                continue;
            }
            crow = cf.D + cf.dbase[r] + (c - cf.cfgbase[r]);
            cstride = cf.ncfg[r];
            atomicAdd(&cf.cfg_net[c], 1);
            if (SITES && cf.cfg_sites) keep_site(env, 2, c, item_index, (u32)pi, i, L, (int)hs);
        } else {
            crow = env->ct->C + (env->ct->cbase[r] - env->ct->cbase0) + (u64)g * pt.n_pid * nk;
            if (mode == 1) {
                const u32 rr = r - env->rh->r0;
                u32 slot = atomicAdd(&env->rh->cnt[rr], 1u);
                if (slot < env->rh->capr) {
                    env->rh->buf[(u64)rr * env->rh->capr + slot] = RefHit{r, (int)hs, L, pl};
                    if (SITES) keep_site(env, 1, (u64)rr * env->rh->capr + slot, item_index, (u32)pi, i, L, (int)hs);
                } else {
                    st->refhit_overflow = 1;
                }
            } else {
                ++counted;
            }
        }
        for (u32 k = 0; k < nk; ++k) {
            i64 is = inner[k].start - region_start, ie = inner[k].end - region_start;
            bool ov = (hs >= is && hs <= ie) || (he >= is && he <= ie);  // inner.overlaps(match.range), range.rs:18-21
            if (ov) atomicAdd(&crow[((size_t)pl * nk + k) * cstride], inner[k].multiplicity);
        }
        if (env->mt->enabled) {
            u64 slot = atomicAdd(&st->n_matches, 1ULL);
            if (slot < env->mt->cap) {
                env->mt->region[slot] = r;
                env->mt->pattern_index[slot] = (u32)pi;
                env->mt->group[slot] = g;
                env->mt->start[slot] = region_start + hs;
            }
        }
    }
    return counted;
}

// Sum of the G table words of one triple, as a balanced tree (short dependency chains).
template <int LO, int HI>
__device__ __forceinline__ u64 pair_sum(const u8* tb, const u32 (&idx)[kMaxGroups]) {
    if constexpr (HI - LO == 1) {
        return *reinterpret_cast<const u64*>(tb + LO * (kPairEntries * 8) + idx[LO]);
    } else {
        constexpr int MID = (LO + HI) / 2;
        return pair_sum<LO, MID>(tb, idx) + pair_sum<MID, HI>(tb, idx);
    }
}

// All triples of one run (same number of column pairs G): G LDS.64 + 64-bit adds per triple and lane.
template <int G, int FIELDS, bool SITES>
__device__ __forceinline__ void scan_run(const u8* tb, u32 n_trip, u32 t0, const u32 (&idx)[kMaxGroups], u32 i, u32 item_index,
                                         const ChunkDesc& cd, const ScanEnv* env, u32& n_counted) {
#pragma unroll SCAN_UNROLL
    for (u32 t = 0; t < n_trip; ++t) {
        u64 acc = pair_sum<0, G>(tb, idx);
        u64 hit = acc & HitMask<FIELDS>::value;
        if (hit && i != 0xffffffffu) n_counted += scan_on_hit<SITES>(hit, t0 + t, i, item_index, cd, env);
        tb += G * (kPairEntries * 8);
    }
}

template <int FIELDS, bool SITES>
__device__ __forceinline__ void scan_dispatch(u32 G, const u8* tb, u32 n_trip, u32 t0, const u32 (&idx)[kMaxGroups], u32 i, u32 item_index,
                                              const ChunkDesc& cd, const ScanEnv* env, u32& n_counted) {
    switch (G) {
#define TFBS_CASE(N) case N: scan_run<N, FIELDS, SITES>(tb, n_trip, t0, idx, i, item_index, cd, env, n_counted); break;
        TFBS_CASE(1) TFBS_CASE(2) TFBS_CASE(3) TFBS_CASE(4) TFBS_CASE(5) TFBS_CASE(6) TFBS_CASE(7) TFBS_CASE(8)
        TFBS_CASE(9) TFBS_CASE(10) TFBS_CASE(11) TFBS_CASE(12) TFBS_CASE(13) TFBS_CASE(14) TFBS_CASE(15) TFBS_CASE(16)
#undef TFBS_CASE
    }
}

__device__ __forceinline__ u32 pair_code_bytes(u32 a, u32 b) {  // pair_entry(a, b) * 8
    u32 e = (a < 4 && b < 4) ? 4 * a + b : (a == 4 ? 16 + b : 21 + a);
    return e * 8;
}


// One launch per pattern chunk.  Persistent CTAs (one per SM) hold the chunk's tables in shared memory; every WARP
// takes `per_grab` consecutive entries of the list from an atomic counter, stages their packed bases into its private
// pair-code planes (several short items side by side, long items in tiles) and scans all triples of the chunk, 32 window
// starts at a time.
template <int FIELDS, bool SITES = false>
__global__ void __launch_bounds__(SCAN_CTA, 1)
    k_scan(const __grid_constant__ DevBlock b, const __grid_constant__ DevSeqs sq, const __grid_constant__ DevPatterns pt,
           const __grid_constant__ DevCounts ct, const __grid_constant__ DevMatches mt, const __grid_constant__ DevRefHits rh,
           const __grid_constant__ DevConfigs cf, int use_cf, const u32* list, const u64* n_list_ptr, u32 per_grab, DevStatus* st,
           u32 chunk) {
    if (use_cf && cf.plan->abort) return;  // an earlier stage ran out of scratch: the host repeats the run
    TFBS_DYNAMIC_SHARED(smem_raw);
    CtaShared* cs = reinterpret_cast<CtaShared*>(smem_raw);
    WarpShared* ws = reinterpret_cast<WarpShared*>(smem_raw + sizeof(CtaShared)) + (threadIdx.x >> 5);
    u8* tbl = smem_raw + sizeof(CtaShared) + SCAN_WARPS * sizeof(WarpShared);
    const u32 tid = threadIdx.x, lane = tid & 31;
    const ChunkDesc cd = pt.chunks[chunk];
    {  // tables: 128-bit coalesced copies (chunks are 16-byte aligned and padded)
        const uint4* src = reinterpret_cast<const uint4*>(pt.table + cd.tbl_off);
        uint4* dst = reinterpret_cast<uint4*>(tbl);
        u32 n16 = (cd.tbl_words + 1) / 2;
        for (u32 k = tid; k < n16; k += SCAN_CTA) dst[k] = src[k];
        if (tid < cd.n_runs && tid < MAX_RUNS) cs->runs[tid] = pt.runs[cd.run_off + tid];
        if (tid == 0) {
            cs->n_runs = cd.n_runs;
            // entries per trip to the work counter: `per_grab` when the list is long, fewer when every warp would otherwise get only
            // one or two trips (a short list, e.g. one rank's shard of a strong-scaled block): the last trips decide the tail
            const u64 n_list = *n_list_ptr;
            const u64 per_warp = n_list / ((u64)gridDim.x * SCAN_WARPS * 6) + 1;
            cs->per_grab = per_warp < per_grab ? (u32)per_warp : per_grab;
            cs->n_list = n_list;
        }
    }
    __syncthreads();
    const u32 n_runs = cs->n_runs;
    const ScanEnv env{use_cf ? &cf : nullptr, &b, &sq, &pt, &ct, &mt, &rh, st};  // for the rare path: pointers to the kernel's own parameters

    for (;;) {
        u32 w = 0;
        if (lane == 0) w = atomicAdd(&st->work_counter, 1u);
        w = __shfl_sync(0xffffffffu, w, 0);
        u64 li = (u64)w * cs->per_grab;
        if (li >= cs->n_list) break;
        const u64 lend = li + cs->per_grab < cs->n_list ? li + cs->per_grab : cs->n_list;
        u32 done_in_item = 0;  // starts of entry li already scored
        u32 n_counted = 0;
        while (li < lend) {
            __syncwarp();
            // a round: pack entries (long items in tiles of TILE_POS starts) into the planes until they are full
            u32 np = 0, pos_used = 0, vtot = 0;
            while (li < lend && np < MAX_PIECES) {
                const u32 item_index = list[li];
                const ScanItem item = sq.items[item_index];
                const u32 q = item.q;
                const u32 len = sq.seq_len[q];
                const u32 left = item.p1 - item.p0 + 1 - done_in_item;
                const u32 n = left < (u32)TILE_POS ? left : (u32)TILE_POS;
                const u32 blk = (n + 32 + 31) & ~31u;
                if (pos_used + blk > 2 * (PLANE_BYTES - 16) && np > 0) break;
                const u32 p0 = item.p0 + done_in_item;
                if (lane == 0) { ws->piece_p0[np] = p0; ws->piece_vstart[np] = vtot; ws->piece_pbase[np] = pos_used; ws->piece_item[np] = item_index; }
                {   // stage this piece: packed bases of [p0, p0 + blk + 1) -> pair codes at plane positions pos_used ..
                    const u64* gpk = sq.pk + sq.ent_uoff[li];
                    const u32* gnm = sq.nm + sq.ent_uoff[li];
                    const u32 n_units = sq.ent_units[li];
                    const u32 u0 = p0 / 32 - item.p0 / 32, o = p0 & 31;
                    const u32 nu = (o + blk + 1) / 32 + 1;
                    __syncwarp();
                    for (u32 k = lane; k < nu; k += 32) {
                        bool in = u0 + k < n_units;
                        ws->raw_pk[k] = in ? gpk[u0 + k] : 0ULL;
                        ws->raw_nm[k] = in ? gnm[u0 + k] : 0xffffffffu;
                    }
                    __syncwarp();
                    for (u32 j = lane; j < blk; j += 32) {
                        u32 x0 = o + j, x1 = x0 + 1;
                        u32 a = (u32)(ws->raw_pk[x0 >> 5] >> (2 * (x0 & 31))) & 3u;
                        u32 bb = (u32)(ws->raw_pk[x1 >> 5] >> (2 * (x1 & 31))) & 3u;
                        if (((ws->raw_nm[x0 >> 5] >> (x0 & 31)) & 1u) || p0 + j >= len) a = 4;
                        if (((ws->raw_nm[x1 >> 5] >> (x1 & 31)) & 1u) || p0 + j + 1 >= len) bb = 4;
                        const u32 jj = pos_used + j;
                        ws->plane[jj & 1][jj >> 1] = (u8)pair_code_bytes(a, bb);
                    }
                }
                pos_used += blk;
                vtot += n;
                ++np;
                done_in_item += n;
                if (done_in_item == item.p1 - item.p0 + 1) { ++li; done_in_item = 0; }
            }
            if (lane == 0) { ws->piece_vstart[np] = vtot; ws->n_pieces = np; }
            __syncwarp();
            for (u32 v0 = 0; v0 < vtot; v0 += 32) {
                const u32 v = v0 + lane;
                u32 k = 0;
                while (k + 1 < np && v >= ws->piece_vstart[k + 1]) ++k;
                const bool valid = v < vtot;
                const u32 off = valid ? v - ws->piece_vstart[k] : 0u;
                const u32 j = ws->piece_pbase[k] + off;
                const u32 i = valid ? ws->piece_p0[k] + off : 0xffffffffu;
                const u32 item_index = ws->piece_item[k];
                const u8* pl = &ws->plane[j & 1][j >> 1];
                u32 idx[kMaxGroups];
#pragma unroll
                for (int gg = 0; gg < kMaxGroups; ++gg) idx[gg] = pl[gg];
                const u8* tb = tbl;
                u32 t0 = 0;
                for (u32 rn = 0; rn < n_runs; ++rn) {
                    const RunDesc rd = cs->runs[rn];
                    scan_dispatch<FIELDS, SITES>(rd.groups, tb, rd.n_triples, t0, idx, i, item_index, cd, &env, n_counted);
                    tb += (size_t)rd.n_triples * rd.groups * (kPairEntries * 8);
                    t0 += rd.n_triples;
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) n_counted += __shfl_xor_sync(0xffffffffu, n_counted, o);
        if (lane == 0 && n_counted) atomicAdd(&st->n_hits, (u64)n_counted);
    }
}

}  // namespace tfbs
