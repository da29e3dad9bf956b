// k0_grouping.cuh -- K0: grouping of haplotypes by their Vec<Diff> (haplotype.rs:65-75)
// Part of the sm_100a kernels of the find-tfbs hot path; included through kernels.cuh (see the map there).
#pragma once
#include "dev_common.cuh"

namespace tfbs {

// ------------------------------------------------------------------------------------------------
// K0: grouping of haplotypes by their Vec<Diff> (haplotype.rs:65-75)
// ------------------------------------------------------------------------------------------------

__device__ __forceinline__ bool same_diff(const DevBlock& b, const tfbs_variant& x, const tfbs_variant& y) {
    if (x.pos != y.pos || x.ref_len != y.ref_len || x.alt_len != y.alt_len) return false;
    for (u32 i = 0; i < x.ref_len; ++i)
        if (b.allele_codes[x.ref_off + i] != b.allele_codes[y.ref_off + i]) return false;
    for (u32 i = 0; i < x.alt_len; ++i)
        if (b.allele_codes[x.alt_off + i] != b.allele_codes[y.alt_off + i]) return false;
    return true;
}

// One CTA per region.  Two records with equal (pos, reference, alternative) are the same Diff value
// for Vec<Diff> equality, so they share a class.
__global__ void k_variant_prep(DevBlock b, u32 r0, u32* var_class, u8* var_inwin, u32* region_dups) {
    u32 r = r0 + blockIdx.x;
    u32 v0 = b.var_off[r], v1 = b.var_off[r + 1];
    i64 s = b.region_start[r], e = b.region_end[r];
    if (region_dups && threadIdx.x == 0) region_dups[r] = 0;
    __syncthreads();
    for (u32 v = v0 + threadIdx.x; v < v1; v += blockDim.x) {
        tfbs_variant x = b.variants[v];
        var_inwin[v] = (x.pos >= s && x.pos <= e) ? 1 : 0;
        u32 cls = v - v0;
        for (u32 u = v0; u < v; ++u)
            if (same_diff(b, b.variants[u], x)) { cls = u - v0; break; }
        var_class[v] = cls;
        if (region_dups && cls != v - v0) region_dups[r] = 1;
        if (b.var_row_out) b.var_row_out[v] = x.carrier_row;
        if (b.var_althash) {  // patch_haplotype gives every ALT base the record's position (haplotype.rs:130-132,136-137)
            u64 a = 0, pw = 1;
            for (u32 t = 0; t < x.alt_len; ++t) { a += hash_val(b.allele_codes[x.alt_off + t], (int)(x.pos - s), b.hash_seed) * pw; pw *= HASH_B; }
            b.var_althash[v] = a;
        }
    }
}

// words of carried-record masks per region: H * ceil(V / 32)
__global__ void k_mask_words(DevBlock b, u32* words) {
    const u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < b.R) words[r] = b.H * ((b.var_off[r + 1] - b.var_off[r] + 31) / 32);
}

__device__ __forceinline__ bool carries(const DevBlock& b, u32 v, u32 h) {
    return (b.carriers[(size_t)b.variants[v].carrier_row * b.pitch + (h >> 5)] >> (h & 31)) & 1u;
}

// Transpose of a 32 x 32 bit matrix held one row per lane: lane l returns column l (bit j = bit l of lane j's row); five butterfly
// exchanges.
__device__ __forceinline__ u32 warp_transpose32(u32 a, u32 lane) {
    u32 m = 0x0000ffffu;
#pragma unroll
    for (u32 j = 16; j; j >>= 1, m ^= m << j) {
        const u32 other = __shfl_xor_sync(0xffffffffu, a, j);
        if ((lane & j) == 0) a ^= (((a >> j) ^ other) & m) << j;
        else a ^= ((other >> j) ^ a) & m;
    }
    return a;
}

// Warp per (region, 32 consecutive haplotypes), lane = haplotype: hash of the ordered list of carried Diff classes; 0 = no diff
// (such a haplotype stays in the reference set, main.rs:74-81,103-105).  Launch with nr * ceil(H / 32) * 32 threads.
// sig_mask: ~0 except under option test_sig_bits (testing), which keeps a few bits of the first attempt's signatures so that different
// diff lists share one and the exact check must catch it.
__global__ void k_signatures(DevBlock b, u32 r0, u32 nr, u64 seed, u64 sig_mask, u64* sig, u32* nd_in) {
    const u64 idx = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u32 HW = (b.H + 31) / 32, lane = threadIdx.x & 31;
    const u64 wg = idx >> 5;
    if (wg >= (u64)nr * HW) return;  // whole warps leave together
    const u32 r = r0 + (u32)(wg / HW), hw = (u32)(wg % HW), h = hw * 32 + lane;
    const bool valid = h < b.H;
    u64 s = seed;
    u32 carried = 0, inw = 0;
    const u32 v0 = b.var_off[r], v1 = b.var_off[r + 1];
    if (b.hap_mask) {
        // first the mask, 32 records per word: lane j fetches the carrier word of record vb + j for these 32 haplotypes (one load
        // instruction for 32 records), a bit-matrix transpose turns record-major into haplotype-major; then the hash over the set
        // bits: a haplotype carries a few records out of dozens
        u32* mask = b.hap_mask + b.mask_base[r] + h;  // word w of haplotype h sits at w * H + h: a warp writes 32 consecutive words
        for (u32 vb = v0, w = 0; vb < v1; vb += 32, ++w) {
            const u32 v = vb + lane;
            const u32 cw = v < v1 ? b.carriers[(size_t)b.var_row[v] * b.pitch + hw] : 0u;
            const u32 word = warp_transpose32(cw, lane);
            if (!valid) continue;
            mask[(u64)w * b.H] = word;
            for (u32 m = word; m; m &= m - 1) {
                const u32 vv = vb + (u32)__ffs((int)m) - 1;
                s = mix64(s + b.var_class[vv] + 1) * 0x9e3779b97f4a7c15ULL + carried;
                ++carried;
                inw += b.var_inwin[vv];
            }
        }
    } else if (valid) {
        for (u32 v = v0; v < v1; ++v)
            if (carries(b, v, h)) {
                s = mix64(s + b.var_class[v] + 1) * 0x9e3779b97f4a7c15ULL + carried;
                ++carried;
                inw += b.var_inwin[v];
            }
    }
    if (!valid) return;
    sig[(size_t)r * b.H + h] = carried ? ((mix64(s) & sig_mask) | 1ULL) : 0ULL;
    nd_in[(size_t)r * b.H + h] = inw;
}

__device__ __forceinline__ u32 table_find_or_insert(u64* keys, u32 mask, u64 key) {
    u32 slot = (u32)(key >> 17) & mask;
    for (;;) {
        u64 prev = atomicCAS(&keys[slot], 0ULL, key);
        if (prev == 0ULL || prev == key) return slot;
        slot = (slot + 1) & mask;
    }
}
__device__ __forceinline__ u32 table_find(const u64* keys, u32 mask, u64 key) {
    u32 slot = (u32)(key >> 17) & mask;
    for (;;) {
        u64 k = keys[slot];
        if (k == key) return slot;
        if (k == 0ULL) return 0xffffffffu;
        slot = (slot + 1) & mask;
    }
}

__device__ __forceinline__ u64 region_key(u64 h, u32 r) { return mix64(h ^ ((u64)(r + 1) * 0xd6e8feb86659fd93ULL)) | 1ULL; }

// seg > 0: the table is cut into one segment of `seg` slots (a power of two >= 2 * H) per region of the batch, so that the slots a
// region touches stay in L2 while its haplotypes are inserted and looked up; seg == 0: one table of mask + 1 slots for the batch.
__global__ void k_group_insert(u32 H, u32 r0, u32 nr, const u64* sig, u64* keys, u32* vals, u32 mask, u32 seg) {
    u64 idx = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (u64)nr * H) return;
    u32 r = r0 + (u32)(idx / H), h = (u32)(idx % H);
    u64 s = sig[(size_t)r * H + h];
    if (!s) return;
    const u64 base = seg ? (u64)(r - r0) * seg : 0;
    u32 slot = table_find_or_insert(keys + base, seg ? seg - 1 : mask, region_key(s, r));
    atomicMin(&vals[base + slot], h);
}

// leader[r,h] = smallest haplotype with the same signature; the class lists are compared exactly so
// that a hash collision is detected (and retried with another seed) instead of merging two groups.
__global__ void k_group_lookup(DevBlock b, u32 r0, u32 nr, const u64* sig, const u64* keys, const u32* vals, u32 mask, u32 seg, u32* leader,
                               DevStatus* st) {
    u64 idx = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (u64)nr * b.H) return;
    u32 r = r0 + (u32)(idx / b.H), h = (u32)(idx % b.H);
    u64 s = sig[(size_t)r * b.H + h];
    if (!s) { leader[(size_t)r * b.H + h] = 0xffffffffu; return; }
    const u64 base = seg ? (u64)(r - r0) * seg : 0;
    u32 slot = table_find(keys + base, seg ? seg - 1 : mask, region_key(s, r));
    u32 ld = vals[base + slot];
    leader[(size_t)r * b.H + h] = ld;
    if (ld == h) return;
    bool ok = ld < b.H;
    if (ok && b.hap_mask) {  // equal masks = the same records = equal lists; different masks are different lists unless the region holds duplicates
        const u32 nw = (b.var_off[r + 1] - b.var_off[r] + 31) / 32;
        const u32* mr = b.hap_mask + b.mask_base[r];
        bool same = true;
        for (u32 w = 0; w < nw && same; ++w) same = mr[(u64)w * b.H + h] == mr[(u64)w * b.H + ld];
        if (same) return;
        if (!b.region_dups[r]) { atomicAdd(&st->sig_collision, 1u); return; }
    }
    if (ok) {
        u32 v1 = b.var_off[r + 1];
        u32 i = b.var_off[r], j = i;
        for (;;) {
            while (i < v1 && !carries(b, i, h)) ++i;
            while (j < v1 && !carries(b, j, ld)) ++j;
            if (i == v1 || j == v1) { ok = (i == v1 && j == v1); break; }
            if (b.var_class[i] != b.var_class[j]) { ok = false; break; }
            ++i; ++j;
        }
    }
    if (!ok) atomicAdd(&st->sig_collision, 1u);
}

// One CTA per region: groups are numbered 1.. in order of their smallest haplotype; 0 is the reference.
__global__ void k_group_rank(u32 H, u32 r0, const u32* leader, const u32* nd_in, u32* hap_group, u32* ngroups, u32* sum_nd) {
    __shared__ u32 s_warp[32];
    __shared__ u32 s_base;
    __shared__ u32 s_nd;
    u32 r = r0 + blockIdx.x;
    const u32* ld = leader + (size_t)r * H;
    u32* hg = hap_group + (size_t)r * H;
    if (threadIdx.x == 0) { s_base = 0; s_nd = 0; }
    __syncthreads();
    u32 lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (u32 h0 = 0; h0 < H; h0 += blockDim.x) {
        u32 h = h0 + threadIdx.x;
        u32 flag = (h < H && ld[h] == h) ? 1u : 0u;
        u32 bal = __ballot_sync(0xffffffffu, flag);
        u32 pre = __popc(bal & ((1u << lane) - 1));
        if (lane == 0) s_warp[wid] = __popc(bal);
        __syncthreads();
        u32 woff = 0, tot = 0;
        for (u32 w = 0; w < nw; ++w) { u32 c = s_warp[w]; if (w < wid) woff += c; tot += c; }
        u32 base = s_base;
        if (flag) {
            hg[h] = 1 + base + woff + pre;
            atomicAdd(&s_nd, nd_in[(size_t)r * H + h]);
        }
        __syncthreads();
        if (threadIdx.x == 0) s_base = base + tot;
        __syncthreads();
    }
    for (u32 h = threadIdx.x; h < H; h += blockDim.x) {
        u32 l = ld[h];
        if (l == 0xffffffffu) hg[h] = 0;
        else if (l != h) hg[h] = hg[l < H ? l : h];  // leaders were written above
    }
    if (threadIdx.x == 0) { ngroups[r] = 1 + s_base; sum_nd[r] = s_nd; }
}

// ---- K0 with the region in shared memory: k_signatures + k_group_insert + k_group_lookup + k_group_rank in one CTA per region ----
// The same signatures, leaders (smallest haplotype of a signature), collision checks and group numbers; nothing but the results
// leaves the CTA.  Dynamic shared memory: the table (u64 key + u32 smallest haplotype per slot, `slots` a power of two > H), per
// haplotype its slot (then its leader) and its in-window record count (then, at leaders, its group), and the masks.
constexpr u32 GROUP_REGION_THREADS = 1024;
constexpr u32 GROUP_REGION_BATCH = 4;  // carrier words a lane loads before it transposes them: independent loads in flight
__host__ __device__ __forceinline__ u64 group_region_smem(u32 H, u32 slots, u32 max_words) {
    return (u64)slots * 12 + (u64)H * 8 + (u64)H * max_words * 4;
}

// Writes hap_group, ngroups and sum_nd like k_group_rank, the masks of the leaders only (k_walk reads nothing else), and per group
// g >= 1 its leader and in-window record count at grp_leader / grp_nd[r * H + g - 1] (k_seq_init_groups).
__global__ void __launch_bounds__(GROUP_REGION_THREADS, 1)
k_group_region(DevBlock b, u64 seed, u64 sig_mask, u32 slots, u32* hap_group, u32* ngroups, u32* sum_nd, u32* grp_leader, u32* grp_nd, DevStatus* st) {
    TFBS_DYNAMIC_SHARED(smem_raw);
    __shared__ u32 s_warp[32];
    __shared__ u32 s_base, s_nd;
    const u32 r = blockIdx.x, H = b.H, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nwarp = blockDim.x >> 5;
    const u32 v0 = b.var_off[r], v1 = b.var_off[r + 1], nw = (v1 - v0 + 31) / 32, HW = (H + 31) / 32, tmask = slots - 1;
    u64* s_key = (u64*)smem_raw;
    u32* s_val = (u32*)(s_key + slots);
    u32* s_ref = s_val + slots;  // slot of the haplotype's signature (0xffffffff: no diff), then its leader
    u32* s_cnt = s_ref + H;      // in-window records carried, then at leaders the group number
    u32* s_mask = s_cnt + H;     // word w of haplotype h at w * H + h
    for (u32 i = tid; i < slots; i += blockDim.x) { s_key[i] = 0; s_val[i] = 0xffffffffu; }
    if (tid == 0) { s_base = 0; s_nd = 0; }
    __syncthreads();

    // signatures (k_signatures: warp per 32 haplotypes, lane = haplotype), inserted as soon as they are known
    for (u32 hw = wid; hw < HW; hw += nwarp) {
        const u32 h = hw * 32 + lane;
        const bool valid = h < H;
        u64 s = seed;
        u32 carried = 0, inw = 0;
        for (u32 w0 = 0; w0 < nw; w0 += GROUP_REGION_BATCH) {
            u32 cw[GROUP_REGION_BATCH];
#pragma unroll
            for (u32 i = 0; i < GROUP_REGION_BATCH; ++i) {
                const u32 v = v0 + (w0 + i) * 32 + lane;
                cw[i] = (w0 + i < nw && v < v1) ? b.carriers[(size_t)b.var_row[v] * b.pitch + hw] : 0u;
            }
#pragma unroll
            for (u32 i = 0; i < GROUP_REGION_BATCH; ++i) {
                if (w0 + i >= nw) break;  // uniform across the warp
                __syncwarp();             // the lanes leave the bit loop below at different times: all 32 meet at the transpose
                const u32 word = warp_transpose32(cw[i], lane);
                if (valid) {
                    s_mask[(w0 + i) * H + h] = word;
                    const u32 vb = v0 + (w0 + i) * 32;
                    for (u32 m = word; m; m &= m - 1) {
                        const u32 vv = vb + (u32)__ffs((int)m) - 1;
                        s = mix64(s + b.var_class[vv] + 1) * 0x9e3779b97f4a7c15ULL + carried;
                        ++carried;
                        inw += b.var_inwin[vv];
                    }
                }
            }
        }
        if (!valid) continue;  // no shuffle follows in this warp's last word of haplotypes
        s_cnt[h] = inw;
        u32 slot = 0xffffffffu;
        if (carried) {
            slot = table_find_or_insert(s_key, tmask, (mix64(s) & sig_mask) | 1ULL);
            atomicMin(&s_val[slot], h);
        }
        s_ref[h] = slot;
    }
    __syncthreads();

    // leaders and their exact check (k_group_lookup); a leader's mask goes out for k_walk
    u32* gmask = b.hap_mask + b.mask_base[r];
    for (u32 h = tid; h < H; h += blockDim.x) {
        const u32 slot = s_ref[h];
        const u32 ld = slot == 0xffffffffu ? 0xffffffffu : s_val[slot];
        s_ref[h] = ld;
        if (ld == h) {
            for (u32 w = 0; w < nw; ++w) gmask[(u64)w * H + h] = s_mask[w * H + h];
            continue;
        }
        if (ld == 0xffffffffu) continue;
        bool same = true;
        for (u32 w = 0; w < nw && same; ++w) same = s_mask[w * H + h] == s_mask[w * H + ld];
        if (same) continue;
        if (b.region_dups[r]) {  // different records may still be the same Diff values: compare the class lists
            u32 wi = 0, wj = 0, mi = nw ? s_mask[h] : 0u, mj = nw ? s_mask[ld] : 0u;
            for (;;) {
                while (!mi && ++wi < nw) mi = s_mask[wi * H + h];
                while (!mj && ++wj < nw) mj = s_mask[wj * H + ld];
                if (!mi || !mj) { same = !mi && !mj; break; }
                const u32 vi = v0 + wi * 32 + (u32)__ffs((int)mi) - 1, vj = v0 + wj * 32 + (u32)__ffs((int)mj) - 1;
                if (b.var_class[vi] != b.var_class[vj]) break;
                mi &= mi - 1;
                mj &= mj - 1;
            }
        }
        if (!same) atomicAdd(&st->sig_collision, 1u);
    }
    __syncthreads();

    // groups numbered 1.. in order of their leader (k_group_rank)
    u32* hg = hap_group + (size_t)r * H;
    u32 nd_part = 0;
    for (u32 h0 = 0; h0 < H; h0 += blockDim.x) {
        const u32 h = h0 + tid;
        const u32 flag = (h < H && s_ref[h] == h) ? 1u : 0u;
        const u32 bal = __ballot_sync(0xffffffffu, flag);
        if (lane == 0) s_warp[wid] = __popc(bal);
        __syncthreads();
        u32 woff = 0, tot = 0;
        for (u32 w = 0; w < nwarp; ++w) { const u32 c = s_warp[w]; if (w < wid) woff += c; tot += c; }
        const u32 base = s_base;
        if (flag) {
            const u32 g = 1 + base + woff + __popc(bal & ((1u << lane) - 1));
            const u32 nd = s_cnt[h];
            hg[h] = g;
            grp_leader[(size_t)r * H + g - 1] = h;
            grp_nd[(size_t)r * H + g - 1] = nd;
            nd_part += nd;
            s_cnt[h] = g;
        }
        __syncthreads();
        if (tid == 0) s_base = base + tot;
    }
    if (nd_part) atomicAdd(&s_nd, nd_part);
    __syncthreads();
    for (u32 h = tid; h < H; h += blockDim.x) {
        const u32 ld = s_ref[h];
        if (ld == 0xffffffffu) hg[h] = 0;
        else if (ld != h) hg[h] = s_cnt[ld];
    }
    if (tid == 0) { ngroups[r] = 1 + s_base; sum_nd[r] = s_nd; }
}

}  // namespace tfbs
