// k3_fanout.cuh -- K3, configuration path: count differences -> per-haplotype-group counts -> min/max filter -> grouped rows
// Part of the sm_100a kernels of the find-tfbs hot path; included through kernels.cuh (see the map there).
//
// count_matches_by_sample (main.rs:500-534) gives every sample the hits of its two haplotypes; here a haplotype's count for a key
// (pattern_id, inner region) is the reference haplotype's count plus the differences of its live configurations.  One warp owns a key:
// it builds the count of every distinct haplotype (group) of the region in a shared-memory vector, then takes min and max of
// left + right over the samples (main.rs:441-451) and, if the key is kept (min != max, main.rs:456-458), writes ONE GROUPED ROW:
// the count of every group, as `bits`-wide offsets from the row's smallest count.  The region's haplotype -> group map goes to the
// host once per region, not once per row: identical count vectors are stored once.
//
// Where the count vector lives.  k_fanout<false> keeps it in dynamic shared memory: 53,120 groups fit next to the pairs, the staging
// buffer and the kernel's static shared memory (227 KB a block on sm_100).  A region of a dense biobank cohort has more distinct haplotypes than that (nearly every one of its 2 x samples
// haplotypes), so k_fanout<true> keeps it in device memory instead, a slice of `groups_cap` words per CTA: capacity is the only reason.
// Per key the vector sees a few hundred touched groups (sparse path) or one pass over the region's groups (dense path), and the sample
// loop's random reads hit L2 as long as the grid's slices fit in its 126 MB (148 SMs x FAN_VEC_CTAS_PER_SM slices).  That variant runs
// a fixed grid whose CTAs walk the (region, CTA of the region) units of dim3(R, split) in a grid-stride loop and own one slice each for
// the whole launch; the kernel leaves the vector all zero after every key, so one memset of the slices per run is enough (a fresh or
// regrown allocation is not zero).
#pragma once
#include "k2c_configs.cuh"

namespace tfbs {

struct DevFan {
    const u32* hap_group;   // [R][H]
    const u64* gbase;       // groups of region r = gbase[r + 1] - gbase[r]
    u32 n_pid;
    int rows_mode;
    u32 groups_cap;         // groups the per-warp count vector holds
    // per key
    u32* vmin;
    u32* vmax;
    u32* flag;              // 1 = the key becomes a row
    u32* k_base;            // smallest per-group count of the key's row
    u8* k_bits;             // width of a packed entry
    u64* k_off;             // first packed word of the row
    const u64* rowidx;      // exclusive scan of flag (k_row_headers)
    // rows
    u64 rows_cap, words_cap;
    u32* o_region;
    u32* o_inner;
    u16* o_pid;
    u32* o_vmin;
    u32* o_vmax;
    u32* o_base;
    u8* o_bits;
    u64* o_off;
    u32* o_packed;
    const u16* pid_list;
    u32* max_count;         // largest left + right of an emitted row
    u32 hg16;               // 1 = the region's haplotype -> group map is kept in shared memory as u16
    // k_fanout<true> only: the count vectors in device memory (one slice of vec_stride words per CTA, all zero on entry) and the
    // number of CTAs per region the units are cut into
    u32* vec;
    u64 vec_stride;
    u32 split;
};

__device__ __forceinline__ u32 bits_for(u32 span) {  // width that holds 0..span: 0, 1, 2, 4, 8, 16 or 32
    if (span == 0) return 0;
    if (span < 2) return 1;
    if (span < 4) return 2;
    if (span < 16) return 4;
    if (span < 256) return 8;
    if (span < 65536) return 16;
    return 32;
}

// Packs the counts of the 32 consecutive groups [g0, g0 + 32) held by the lanes of a warp (lane l: value v of group g0 + l, 0 behind
// the last group) as `bits`-wide fields: they fill `bits` consecutive words starting at word g0 * bits / 32.  bits is a power of two,
// so the lane -> (word, shift) map is shifts and masks.  Narrow fields (1, 2 bits): word k is the OR over the 32 / bits lanes whose
// group lives in it (REDUX), written by lane k.  Wide fields: a butterfly OR inside each run of 32 / bits lanes, its first lane writes.
__device__ __forceinline__ void pack_32_groups(u32 v, u32 bits, u32 lane, u32* out, u32 n_out) {  // n_out: words of the row left from `out` on
    if (bits == 32) { if (lane < n_out) out[lane] = v; return; }
    const u32 lb = __ffs(bits) - 1, per = 32u >> lb, mine = lane >> (5 - lb);
    u32 x = v << ((lane & (per - 1)) << lb);
    if (bits <= 2) {
        for (u32 k = 0; k < bits; ++k) {
            const u32 word = __reduce_or_sync(0xffffffffu, mine == k ? x : 0u);
            if (lane == k && k < n_out) out[k] = word;
        }
    } else {
        for (u32 o = 1; o < per; o <<= 1) x |= __shfl_xor_sync(0xffffffffu, x, o);
        if ((lane & (per - 1)) == 0 && mine < n_out) out[mine] = x;
    }
}

#ifndef TFBS_FAN_THREADS
#define TFBS_FAN_THREADS 256
#endif
#ifndef TFBS_FAN_PAIRS
#define TFBS_FAN_PAIRS 512
#endif
#ifndef TFBS_FAN_STAGE
#define TFBS_FAN_STAGE 1024
#endif
constexpr int FAN_THREADS = TFBS_FAN_THREADS;
constexpr u32 FAN_PAIRS = TFBS_FAN_PAIRS;    // non-zero (configuration, difference) pairs of a round of FAN_THREADS keys kept in shared memory
constexpr u32 FAN_STAGE = TFBS_FAN_STAGE;    // packed row words staged in shared memory before they are copied out in one piece
constexpr u32 FAN_STAGE_ROWS = 32;
#ifndef TFBS_FAN_SPLIT
#define TFBS_FAN_SPLIT 4
#endif
constexpr u32 FAN_SPLIT = TFBS_FAN_SPLIT;      // smallest number of CTAs per region (gridDim.y): CTA j takes the rounds j, j + gridDim.y, ... of the region's keys
#ifndef TFBS_FAN_VEC_CTAS_PER_SM
#define TFBS_FAN_VEC_CTAS_PER_SM 2
#endif
constexpr u32 FAN_VEC_CTAS_PER_SM = TFBS_FAN_VEC_CTAS_PER_SM;  // k_fanout<true>: grid = SMs x this, one device-memory count vector per CTA

struct FanPair { u32 m0, n, d, cum; };  // members [m0, m0 + n) of the region's member list get the difference d; cum = members of the key's earlier pairs

// Dynamic shared memory of k_fanout<false>: val[groups_cap] | pairs[FAN_PAIRS] | stage[FAN_STAGE] | hg16[H] (if DevFan::hg16);
// k_fanout<true> has no val here (groups_cap = 0)
__host__ __device__ inline size_t fan_smem_bytes(u32 groups_cap, u32 H, bool hg16) {
    return (size_t)groups_cap * 4 + (size_t)FAN_PAIRS * sizeof(FanPair) + (size_t)FAN_STAGE * 4 + (hg16 ? (((size_t)H * 2 + 15) & ~(size_t)15) : 0);
}
// Static shared memory of k_fanout: its __shared__ arrays below (s_scan .. s_base; keep the two in step), rounded up to 128 bytes for
// the padding between them (ptxas -v: 7,648 B).  A block's dynamic shared memory may be what the device allows a block less this.
constexpr size_t FAN_STATIC_SMEM = ((((2 + 4) * (FAN_THREADS / 32) + 4 + 7 * FAN_THREADS + 2 * FAN_STAGE_ROWS) * 4 + 8) + 127) & ~(size_t)127;

// gridDim.y (>= FAN_SPLIT) CTAs per region, each takes every gridDim.y-th round of at most FAN_THREADS keys.
//  A. the round's slab of the difference matrix (FAN_THREADS keys x configurations) is read once, coalesced; the few non-zero
//     entries are counted per key, one block scan gives every key its place, a second pass over the (now cached) slab files the
//     pairs key by key into shared memory.  A key without a non-zero entry -- the large majority: no hit touched it, or what a
//     configuration lost it found again -- has the reference haplotype's count for everybody and is answered at once.
//  B. the remaining keys one at a time, the whole CTA on each: the count of every group is built in ONE count vector (a warp per
//     configuration, lanes over its member groups; two configurations of different clusters can meet in a group, hence atomics),
//     min / max of left + right over the samples are reduced (main.rs:441-451), and when the key becomes a
//     row (min != max, main.rs:456-458) its packed counts are appended to a staging buffer in shared memory while the vector is
//     cleared for the next key.  The staging buffer is copied out in one piece at a position drawn from an atomic cursor -- one
//     global atomic per few dozen rows; the payload order is arbitrary, k_row_headers numbers the rows in key order afterwards.
// VEC = false: CTA (blockIdx.x, blockIdx.y) = unit (region, CTA of the region), count vector in shared memory.
// VEC = true: a fixed grid walks the units of dim3(R, fn.split) in a grid-stride loop, count vector in device memory (see the header).
template <bool VEC>
__global__ void __launch_bounds__(FAN_THREADS) k_fanout(DevBlock b, DevConfigs cf, DevFan fn) {
    TFBS_DYNAMIC_SHARED(smem_raw);
    constexpr u32 NW = FAN_THREADS / 32;
    __shared__ u32 s_scan[2][NW], s_red[4][NW], s_fin[4];
    __shared__ u32 s_cnt[FAN_THREADS], s_fill[FAN_THREADS], s_hkey[FAN_THREADS], s_hfirst[FAN_THREADS], s_hcnt[FAN_THREADS], s_href[FAN_THREADS], s_htot[FAN_THREADS];
    __shared__ u32 s_stage_key[FAN_STAGE_ROWS], s_stage_rel[FAN_STAGE_ROWS];
    __shared__ unsigned long long s_base;
    const u32 tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    // sibling CTAs raise abort while this one runs: one read for the whole CTA, or its threads could part at a barrier below
    if (tid == 0) s_fin[0] = cf.plan->abort;
    __syncthreads();
    if (s_fin[0]) return;
    u32* val = VEC ? fn.vec + (u64)blockIdx.x * fn.vec_stride : reinterpret_cast<u32*>(smem_raw);
    FanPair* pairs = reinterpret_cast<FanPair*>(VEC ? smem_raw : smem_raw + (size_t)fn.groups_cap * 4);
    u32* stage = reinterpret_cast<u32*>(pairs + FAN_PAIRS);
    u16* hg16 = reinterpret_cast<u16*>(stage + FAN_STAGE);
    // (CTAs per region: written out at every use, a variable of its own costs k_fanout<false> registers)
#define TFBS_FAN_SPLIT_NOW (VEC ? fn.split : gridDim.y)
    u32 row_max = 0;
    u32 unit = blockIdx.x;  // VEC: the host's grid has at most R * split < 2^32 CTAs
    do {
        const u32 r = VEC ? unit / fn.split : blockIdx.x;
        const u32 cy = VEC ? unit % fn.split : blockIdx.y;
        if (VEC) __syncthreads();  // the previous unit's map and round arrays are no longer read
        // the keys of the region go to the `split` CTAs in rounds of `rs` keys: equal shares when they fit one round each
        const u32 nkeys_all = fn.n_pid * (b.inner_off[r + 1] - b.inner_off[r]);
        // (a CTA has a fixed cost -- the haplotype -> group map, the zeroed vector -- that only pays when a key is expensive, i.e. when
        // the region has many groups: small regions keep their few keys in one CTA)
        const u32 ng = (u32)(fn.gbase[r + 1] - fn.gbase[r]);
        const u32 kmin = ng >= 8192 ? 1u : (ng >= 1024 ? 16u : 64u);
        const u32 rs = min((u32)FAN_THREADS, max(kmin, (nkeys_all + TFBS_FAN_SPLIT_NOW - 1) / TFBS_FAN_SPLIT_NOW));
        if ((u64)cy * rs >= (u64)nkeys_all) continue;  // no round for this CTA
        if (ng > fn.groups_cap) {  // more distinct haplotypes than the count vector holds: the host repeats the run
            if (tid == 0) { atomicMax(&cf.plan->need[Cap::groups], (u64)ng); cf.plan->abort = 1; }
            return;
        }
        if (tid == 0) atomicMax(&cf.plan->need[Cap::groups], (u64)ng);
        const u32 nk = b.inner_off[r + 1] - b.inner_off[r];
        const u32 nkeys = fn.n_pid * nk;
        const u64 kb = cf.kbase[r];
        const u32 ncfg = cf.ncfg[r];
        const u64 cb = cf.cfgbase[r];
        const u32* Dr = cf.D + cf.dbase[r];
        const u32* hg = fn.hap_group + (size_t)r * b.H;
        const u64 mbase = cf.moff[cb];
        const u32* members = cf.members + mbase;
        if (fn.hg16)
            for (u32 h = tid; h < b.H; h += FAN_THREADS) hg16[h] = (u16)hg[h];
        if (!VEC)  // (the device-memory vectors are zeroed by the host once per run)
            for (u32 g = tid; g < ng; g += FAN_THREADS) val[g] = 0;
        for (u32 w = tid; w < FAN_STAGE; w += FAN_THREADS) stage[w] = 0;  // rows are XORed into the staging buffer: it is all zero between rows
        u32 stage_used = 0, stage_rows = 0;  // the same in every thread: every decision about the staging buffer is uniform

        // copies the staged rows out (all threads); the keys of the staged rows learn their offset
        auto flush = [&]() {
            __syncthreads();
            if (stage_rows) {
                if (tid == 0) s_base = atomicAdd((unsigned long long*)&cf.plan->rowwords_alloc, (unsigned long long)stage_used);
                __syncthreads();
                const u64 base = s_base;
                const bool fits = base + stage_used <= fn.words_cap;  // beyond the capacity: the gate behind this kernel raises abort
                for (u32 w = tid; w < stage_used; w += FAN_THREADS) {
                    if (fits) fn.o_packed[base + w] = stage[w];
                    stage[w] = 0;
                }
                for (u32 i = tid; i < stage_rows; i += FAN_THREADS) fn.k_off[kb + s_stage_key[i]] = base + s_stage_rel[i];
                __syncthreads();
            }
            stage_used = 0;
            stage_rows = 0;
        };

        for (u32 k0 = cy * rs; k0 < nkeys; k0 += TFBS_FAN_SPLIT_NOW * rs) {
            // ---- A: the round's slab of D, coalesced ----
            const u32 nround = nkeys - k0 < rs ? nkeys - k0 : rs;
            const u32* slab = Dr + (u64)k0 * ncfg;
            const u32 nwords = nround * ncfg;
            s_cnt[tid] = 0;
            s_fill[tid] = 0;
            __syncthreads();
            for (u32 i = tid; i < nwords; i += FAN_THREADS)
                if (slab[i]) atomicAdd(&s_cnt[i / ncfg], 1u);
            __syncthreads();
            const u32 key = k0 + tid;
            const u32 cnt = tid < nround ? s_cnt[tid] : 0u;
            const u32 ref_mine = tid < nround ? cf.C0[kb + key] : 0u;
            if (tid < nround && cnt == 0) {
                // every haplotype has the reference haplotype's count: a row only when every key with a hit is asked for (main.rs:517-528)
                const u32 f = (fn.rows_mode == TFBS_ROWS_VARYING || ref_mine == 0) ? 0u : 1u;
                fn.vmin[kb + key] = 2 * ref_mine;
                fn.vmax[kb + key] = 2 * ref_mine;
                fn.flag[kb + key] = f;
                fn.k_base[kb + key] = ref_mine;
                fn.k_bits[kb + key] = 0;
                fn.k_off[kb + key] = 0;
                if (f) row_max = max(row_max, 2 * ref_mine);
            }
            // exclusive block scans: pairs before this key, keys with pairs before this key
            u32 x = cnt, y = cnt ? 1u : 0u;
    #pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const u32 xv = __shfl_up_sync(0xffffffffu, x, o), yv = __shfl_up_sync(0xffffffffu, y, o);
                if (lane >= (u32)o) { x += xv; y += yv; }
            }
            if (lane == 31) { s_scan[0][wid] = x; s_scan[1][wid] = y; }
            __syncthreads();
            u32 xoff = 0, yoff = 0, n_heavy = 0;
            for (u32 w = 0; w < NW; ++w) {
                if (w < wid) { xoff += s_scan[0][w]; yoff += s_scan[1][w]; }
                n_heavy += s_scan[1][w];
            }
            s_hfirst[tid] = 0xffffffffu;  // indexed by key here; re-indexed by heavy position below
            __syncthreads();
            u32 my_first = xoff + x - cnt, my_hpos = yoff + y - 1;
            s_cnt[tid] = my_first;  // first pair of the key (indexed by key - k0), for the filing pass
            __syncthreads();
            for (u32 i = tid; i < nwords; i += FAN_THREADS) {
                const u32 d = slab[i];
                if (!d) continue;
                const u32 kk = i / ncfg, c = i - kk * ncfg;
                const u32 o = s_cnt[kk] + atomicAdd(&s_fill[kk], 1u);
                if (o < FAN_PAIRS) {
                    const u64 m0 = cf.moff[cb + c], m1 = cf.moff[cb + c + 1];
                    pairs[o] = FanPair{(u32)(m0 - mbase), (u32)(m1 - m0), d, 0u};
                }
            }
            if (cnt) {
                s_hkey[my_hpos] = key;
                s_hfirst[my_hpos] = my_first;
                s_hcnt[my_hpos] = cnt;
                s_href[my_hpos] = ref_mine;
            }
            if (tid == 0 && n_heavy) atomicAdd((unsigned long long*)&cf.plan->fan_keys, (unsigned long long)n_heavy);
    #ifdef TFBS_FAN_STATS
            if (tid < n_heavy) { atomicAdd((unsigned long long*)&cf.plan->fan_dbg[0], (unsigned long long)s_hcnt[tid]); }
    #endif
            __syncthreads();
            if (tid < n_heavy && s_hfirst[tid] + s_hcnt[tid] <= FAN_PAIRS) {  // members before every pair of the key: the scatter below is flat
                u32 cum = 0;
                for (u32 j = 0; j < s_hcnt[tid]; ++j) {
                    pairs[s_hfirst[tid] + j].cum = cum;
                    cum += pairs[s_hfirst[tid] + j].n;
                }
                s_htot[tid] = cum;
            }
            __syncthreads();
            // ---- B: the whole CTA per key that needs the count vector (val is all zero on entry) ----
            for (u32 a = 0; a < n_heavy; ++a) {
                const u32 hkey = s_hkey[a], first = s_hfirst[a], hcnt = s_hcnt[a], ref = s_href[a];
                // sparse = the key's pairs sit in shared memory: every later pass visits only the groups a pair touches (a few hundred of
                // the region's thousands), found again through the pairs; the others keep the reference haplotype's count
                const bool sparse = first + hcnt <= FAN_PAIRS;
                const u32 tot = sparse ? s_htot[a] : 0u;
                auto touched = [&](u32 x, u32& d) {  // group of the x-th (configuration, member) of the key
                    u32 j = 0;
                    while (j + 1 < hcnt && pairs[first + j + 1].cum <= x) ++j;
                    const FanPair pr = pairs[first + j];
                    d = pr.d;
                    return members[pr.m0 + (x - pr.cum)];
                };
                u32 g_mine = 0;  // the group of x = tid, kept for the later passes
                if (sparse) {
                    // a thread per (configuration, member group) of the key: two configurations of different clusters can meet in a group
                    for (u32 x = tid; x < tot; x += FAN_THREADS) {
                        u32 d;
                        const u32 g = touched(x, d);
                        if (x == tid) g_mine = g;
                        atomicAdd(&val[g], d);
                    }
                } else {  // more pairs in this round than shared memory holds: this key reads its row again, a lane per configuration;
                          // long member lists are shared out over the warp
                    const u32* drow = Dr + (u64)hkey * ncfg;
                    for (u32 c0 = wid * 32; c0 < ncfg; c0 += NW * 32) {
                        const u32 c = c0 + lane;
                        const u32 d = c < ncfg ? drow[c] : 0u;
                        u64 m0 = 0, m1 = 0;
                        if (d) { m0 = cf.moff[cb + c]; m1 = cf.moff[cb + c + 1]; }
                        const bool longlist = m1 - m0 > 8;
                        if (d && !longlist)
                            for (u64 m = m0; m < m1; ++m) atomicAdd(&val[cf.members[m]], d);
                        u32 todo = __ballot_sync(0xffffffffu, longlist);
                        while (todo) {
                            const int src = __ffs(todo) - 1;
                            todo &= todo - 1;
                            const u64 a0 = __shfl_sync(0xffffffffu, m0, src), a1 = __shfl_sync(0xffffffffu, m1, src);
                            const u32 dd = __shfl_sync(0xffffffffu, d, src);
                            for (u64 m = a0 + lane; m < a1; m += 32) atomicAdd(&val[cf.members[m]], dd);
                        }
                    }
                }
                __syncthreads();
                // smallest / largest count over the groups (the packing base and width), min / max of left + right over the samples
                u32 gmin = ref, gmax = ref, lo = 0xffffffffu, hi = 0;
                if (sparse) {
                    for (u32 x = tid; x < tot; x += FAN_THREADS) {
                        u32 d;
                        const u32 c = ref + val[x == tid ? g_mine : touched(x, d)];
                        gmin = min(gmin, c);
                        gmax = max(gmax, c);
                    }
                } else {
                    for (u32 g = tid; g < ng; g += FAN_THREADS) {
                        const u32 c = ref + val[g];
                        gmin = min(gmin, c);
                        gmax = max(gmax, c);
                    }
                }
    #ifdef TFBS_FAN_STATS
                {
                    u32 tg = 0, ts = 0;
                    for (u32 g = tid; g < ng; g += FAN_THREADS) tg += val[g] != 0;
                    for (u32 s = tid; s < b.S; s += FAN_THREADS) ts += (val[hg[2 * s]] | val[hg[2 * s + 1]]) != 0;
                    atomicAdd((unsigned long long*)&cf.plan->fan_dbg[2], (unsigned long long)tg);
                    atomicAdd((unsigned long long*)&cf.plan->fan_dbg[3], (unsigned long long)ts);
                    if (tid == 0 && first + hcnt <= FAN_PAIRS) atomicAdd((unsigned long long*)&cf.plan->fan_dbg[1], (unsigned long long)s_htot[a]);
                    if (tid == 0 && !sparse) atomicAdd((unsigned long long*)&cf.plan->fan_dbg[4], 1ull);
                }
    #endif
                if (fn.hg16) {
                    for (u32 s = tid; s < b.S; s += FAN_THREADS) {
                        const u32 two = reinterpret_cast<const u32*>(hg16)[s];  // both haplotypes of the sample
                        const u32 v = 2 * ref + val[two & 0xffffu] + val[two >> 16];
                        lo = min(lo, v);
                        hi = max(hi, v);
                    }
                } else {
                    for (u32 s = tid; s < b.S; s += FAN_THREADS) {
                        const u32 v = 2 * ref + val[hg[2 * s]] + val[hg[2 * s + 1]];
                        lo = min(lo, v);
                        hi = max(hi, v);
                    }
                }
    #pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
                    hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
                    gmin = min(gmin, __shfl_xor_sync(0xffffffffu, gmin, o));
                    gmax = max(gmax, __shfl_xor_sync(0xffffffffu, gmax, o));
                }
                if (lane == 0) { s_red[0][wid] = lo; s_red[1][wid] = hi; s_red[2][wid] = gmin; s_red[3][wid] = gmax; }
                __syncthreads();
                if (wid == 0) {  // the first warp reduces the partial results of the warps and publishes the four values
                    lo = lane < NW ? s_red[0][lane] : 0xffffffffu;
                    hi = lane < NW ? s_red[1][lane] : 0u;
                    gmin = lane < NW ? s_red[2][lane] : 0xffffffffu;
                    gmax = lane < NW ? s_red[3][lane] : 0u;
    #pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
                        hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
                        gmin = min(gmin, __shfl_xor_sync(0xffffffffu, gmin, o));
                        gmax = max(gmax, __shfl_xor_sync(0xffffffffu, gmax, o));
                    }
                    if (lane == 0) { s_fin[0] = lo; s_fin[1] = hi; s_fin[2] = gmin; s_fin[3] = gmax; }
                }
                __syncthreads();
                lo = s_fin[0];
                hi = s_fin[1];
                gmin = s_fin[2];
                gmax = s_fin[3];
                // keys exist once a hit of any scanned haplotype touched the inner region (main.rs:517-528): hi > 0
                const u32 f = (fn.rows_mode == TFBS_ROWS_VARYING) ? (lo != hi ? 1u : 0u) : (hi > 0 ? 1u : 0u);
                const u32 bits = bits_for(gmax - gmin);
                const u32 words = (u32)(((u64)ng * bits + 31) / 32);
                if (tid == 0) {
                    fn.vmin[kb + hkey] = lo;
                    fn.vmax[kb + hkey] = hi;
                    fn.flag[kb + hkey] = f;
                    fn.k_base[kb + hkey] = gmin;
                    fn.k_bits[kb + hkey] = (u8)bits;
                    fn.k_off[kb + hkey] = 0;
                }
                if (f) row_max = max(row_max, hi);
                // the row is packed a warp at a time (32 consecutive groups fill `bits` whole words) while the vector is cleared for the next key
                const u32 ng32 = (ng + 31) & ~31u;
                if (f && bits && words <= FAN_STAGE) {
                    if (stage_used + words > FAN_STAGE || stage_rows == FAN_STAGE_ROWS) flush();
                    const u32 rel = stage_used;
                    if (sparse) {
                        // every field holds the reference haplotype's offset, except those of the touched groups: XORed into the zeroed
                        // staging words in any order.  atomicExch hands a group that two pairs touch to one thread and clears the vector.
                        const u32 f0 = ref - gmin;
                        const u32 pat = bits == 32 ? f0 : f0 * (0xffffffffu / ((1u << bits) - 1u));
                        const u32 tail = (ng * bits) & 31u;
                        for (u32 w = tid; w < words; w += FAN_THREADS)
                            atomicXor(&stage[rel + w], (w + 1 == words && tail) ? (pat & ((1u << tail) - 1u)) : pat);
                        for (u32 x = tid; x < tot; x += FAN_THREADS) {
                            u32 d;
                            const u32 g = x == tid ? g_mine : touched(x, d);
                            const u32 old = atomicExch(&val[g], 0u);
                            if (old) atomicXor(&stage[rel + ((g * bits) >> 5)], ((f0 + old) ^ f0) << ((g * bits) & 31u));
                        }
                    } else {
                        for (u32 g = tid; g < ng32; g += FAN_THREADS) {
                            u32 v = 0;
                            if (g < ng) { v = ref + val[g] - gmin; val[g] = 0; }
                            const u32 w0 = (g - lane) / 32 * bits;
                            pack_32_groups(v, bits, lane, stage + rel + w0, words - w0);
                        }
                    }
                    if (tid == 0) { s_stage_key[stage_rows] = hkey; s_stage_rel[stage_rows] = rel; }
                    stage_used = rel + words;
                    stage_rows += 1;
                } else if (f && bits) {  // a row larger than the staging buffer goes out directly
                    if (tid == 0) s_base = atomicAdd((unsigned long long*)&cf.plan->rowwords_alloc, (unsigned long long)words);
                    __syncthreads();
                    const u64 base = s_base;
                    if (tid == 0) fn.k_off[kb + hkey] = base;
                    const bool fits = base + words <= fn.words_cap;
                    for (u32 g = tid; g < ng32; g += FAN_THREADS) {
                        u32 v = 0;
                        if (g < ng) { v = ref + val[g] - gmin; val[g] = 0; }
                        const u32 w0 = (g - lane) / 32 * bits;
                        if (fits) pack_32_groups(v, bits, lane, fn.o_packed + base + w0, words - w0);
                    }
                } else if (sparse) {
                    for (u32 x = tid; x < tot; x += FAN_THREADS) {
                        u32 d;
                        val[x == tid ? g_mine : touched(x, d)] = 0;
                    }
                } else {
                    for (u32 g = tid; g < ng; g += FAN_THREADS) val[g] = 0;
                }
                __syncthreads();
            }
        }
        flush();
    } while (VEC && (unit += gridDim.x) < b.R * fn.split);
#undef TFBS_FAN_SPLIT_NOW
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) row_max = max(row_max, __shfl_xor_sync(0xffffffffu, row_max, o));
    if (lane == 0 && row_max) atomicMax(fn.max_count, row_max);
}

// Rows in key order = (region, pattern_id, inner): thread per key.
__global__ void k_row_headers(DevBlock b, DevConfigs cf, DevFan fn, const u64* n_rows_ptr) {
    if (cf.plan->abort) return;
    const u32 r = blockIdx.x;
    const u32 nk = b.inner_off[r + 1] - b.inner_off[r];
    const u32 nkeys = fn.n_pid * nk;
    const u64 kb = cf.kbase[r];
    for (u32 key = threadIdx.x; key < nkeys; key += blockDim.x) {
        if (!fn.flag[kb + key]) continue;
        const u64 row = fn.rowidx[kb + key];
        if (row >= fn.rows_cap || row >= *n_rows_ptr) continue;
        fn.o_region[row] = r;
        fn.o_inner[row] = b.inner_off[r] + key % nk;
        fn.o_pid[row] = fn.pid_list[key / nk];
        fn.o_vmin[row] = fn.vmin[kb + key];
        fn.o_vmax[row] = fn.vmax[kb + key];
        fn.o_base[row] = fn.k_base[kb + key];
        fn.o_bits[row] = fn.k_bits[kb + key];
        fn.o_off[row] = fn.k_off[kb + key];
    }
}

// Grouped rows -> the reference's (Vec<u32>, Vec<u32>) per key (main.rs:500-534), one warp per row; T = u8 / u16 / u32.
struct DevDenseRows {
    void* left;
    void* right;
};
template <class T>
__global__ void k_rows_expand(u32 S, u32 H, const u32* hap_group, const u64* n_rows_ptr, const u32* o_region, const u32* o_base,
                              const u8* o_bits, const u64* o_off, const u32* o_packed, DevDenseRows out) {
    const u64 row = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const u32 lane = threadIdx.x & 31;
    if (row >= *n_rows_ptr) return;
    const u32* hg = hap_group + (size_t)o_region[row] * H;
    const u32 base = o_base[row], bits = o_bits[row];
    const u32* pk = o_packed + o_off[row];
    const u32 per = bits ? 32 / bits : 0, mask = bits == 32 ? 0xffffffffu : ((1u << bits) - 1);
    T* left = reinterpret_cast<T*>(out.left) + row * S;
    T* right = reinterpret_cast<T*>(out.right) + row * S;
    for (u32 s = lane; s < S; s += 32) {
        const u32 g0 = hg[2 * s], g1 = hg[2 * s + 1];
        left[s] = (T)(base + (bits ? (pk[g0 / per] >> ((g0 % per) * bits)) & mask : 0u));
        right[s] = (T)(base + (bits ? (pk[g1 / per] >> ((g1 % per) * bits)) & mask : 0u));
    }
}

// hap_group as the host gets it with grouped rows: u16 when every region has fewer than 65536 groups
__global__ void k_narrow_groups(const u32* hap_group, u64 n, u16* out) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) out[i] = (u16)hap_group[i];
}

}  // namespace tfbs
