// k1_build.cuh -- K1: haplotype build (patch_haplotype as segments, the sequence-keyed map)
// Part of the sm_100a kernels of the find-tfbs hot path; included through kernels.cuh (see the map there).
#pragma once
#include "dev_common.cuh"
#include "prefix_scan.cuh"
#include "k0_grouping.cuh"

namespace tfbs {

// ------------------------------------------------------------------------------------------------
// K1: haplotype build
// ------------------------------------------------------------------------------------------------

// Window starts [p0, p1] of sequence q.  With delta scoring only the windows that touch a variant are scored for a patched
// haplotype; every other window is identical (bases and positions) to a window of the reference haplotype.
struct __align__(16) ScanItem {
    u32 q, p0, p1;
    u32 index;   // its own index in the work list
};

// A hit of the reference haplotype, kept so that patched haplotypes can inherit or lose it.
struct RefHit {
    u32 region;
    int relpos;   // window start relative to region_start
    u32 len;      // pattern length
    u32 pid;      // pid_index of the pattern
};
struct DevRefHits {
    RefHit* buf;   // slab of `capr` entries per region of the batch
    u32* cnt;      // hits per region of the batch (may exceed capr: then the batch falls back to a full scan)
    u32 capr;
    u32 r0;        // first region of the batch
};

// Sequence table of a batch: q = gbase[r] - gbase[r0] + g.
struct DevSeqs {
    u32 n_seq;               // sequences (an upper bound when n_seq_ptr is set: the count then lives on the device)
    const u64* n_seq_ptr;    // NULL, or the device word that holds the real number of sequences
    const u32* abort;        // NULL, or DevPlan::abort: an earlier stage ran out of scratch, the sequence arrays are not to be trusted
    u32 n_ref;               // > 0: "virtual" sequences of the configuration path: q < n_ref is the reference haplotype of region q,
                             // q >= n_ref a (cluster, carried records) configuration; 0: the distinct haplotypes of the regions
    const u64* gbase;        // per region (block-wide index), first sequence of the region (batch-relative after -gbase0)
    u64 gbase0;
    u32* seq_region;         // [n_seq]
    u32* seq_leader;         // [n_seq] haplotype whose diff list defines the sequence (0xffffffff for the reference)
    u32* seq_nd;             // [n_seq] in-window diffs
    u64* seq_doff;           // [n_seq+1] offset into dlist
    u32* dlist;              // variant indices, sorted per sequence
    Seg* segs;               // at 2*doff + 2*q, at most 2*nd + 2 entries
    u32* seq_nseg;           // [n_seq] segments without the terminator
    u32* seq_len;            // [n_seq] bases
    u32* ent_units;          // [list] packed units of a scored list entry: bases [p0 & ~31, p1 + 64]
    u64* ent_uoff;           // [list+1] offset into pk / nm
    u64* pk;                 // 32 bases per word, 2 bits each
    u32* nm;                 // N mask, bit b = base 32u+b is N
    u64* seq_hash;           // [n_seq]
    u8* seq_flags;           // bit0 truncated, bit1 dropped (overwritten in the sequence-keyed map)
    u32* seq_ntake;          // [n_seq] diffs of dlist the walk consumed: nd, or k + 1 when it was truncated at dlist[k]
    // scan work list: ranges of window starts that have to be scored
    u32* seq_nitems;         // [n_seq]
    u64* item_off;           // [n_seq+1]
    ScanItem* items;         // flat, in sequence order
    u32 n_items_cap;
    u64 units_cap;           // capacity of pk / nm in units (0 = sized exactly, not checked)
};


__device__ __forceinline__ u32 seq_count(const DevSeqs& sq) {  // 0 once the run has been given up
    if (sq.abort && *sq.abort) return 0;
    if (!sq.n_seq_ptr) return sq.n_seq;
    const u64 n = *sq.n_seq_ptr;
    return n < sq.n_seq ? (u32)n : sq.n_seq;
}

__global__ void k_seq_init(u32 H, u32 r0, const u32* hap_group, const u32* leader, const u32* nd_in, DevSeqs sq) {
    u32 r = r0 + blockIdx.x;
    u64 qb = sq.gbase[r] - sq.gbase0;
    if (threadIdx.x == 0 && qb < sq.n_seq) {
        sq.seq_region[qb] = r;
        sq.seq_leader[qb] = 0xffffffffu;
        sq.seq_nd[qb] = 0;
    }
    for (u32 h = threadIdx.x; h < H; h += blockDim.x) {
        if (leader[(size_t)r * H + h] == h) {
            u64 q = qb + hap_group[(size_t)r * H + h];
            if (q >= sq.n_seq) continue;  // more sequences than the scratch holds: the run is repeated (need_seq)
            sq.seq_region[q] = r;
            sq.seq_leader[q] = h;
            sq.seq_nd[q] = nd_in[(size_t)r * H + h];
        }
    }
}
// The same from the per-group lists of k_group_region: group g >= 1 of region r at grp_leader / grp_nd[r * H + g - 1].
__global__ void k_seq_init_groups(u32 H, const u32* ngroups, const u32* grp_leader, const u32* grp_nd, DevSeqs sq) {
    const u32 r = blockIdx.x;
    const u64 qb = sq.gbase[r] - sq.gbase0;
    if (threadIdx.x == 0 && qb < sq.n_seq) {
        sq.seq_region[qb] = r;
        sq.seq_leader[qb] = 0xffffffffu;
        sq.seq_nd[qb] = 0;
    }
    const u32 ng = ngroups[r];
    for (u32 g = 1 + threadIdx.x; g < ng; g += blockDim.x) {
        const u64 q = qb + g;
        if (q >= sq.n_seq) break;  // more sequences than the scratch holds: the run is repeated (need_seq)
        sq.seq_region[q] = r;
        sq.seq_leader[q] = grp_leader[(size_t)r * H + g - 1];
        sq.seq_nd[q] = grp_nd[(size_t)r * H + g - 1];
    }
}

// derived Ord of Diff: (pos, reference, alternative), vectors lexicographic, A<C<G<T<N (types.rs:5-8,39-44)
__device__ __forceinline__ int cmp_codes(const u8* a, u32 na, const u8* b, u32 nb) {
    u32 n = na < nb ? na : nb;
    for (u32 i = 0; i < n; ++i)
        if (a[i] != b[i]) return a[i] < b[i] ? -1 : 1;
    return na == nb ? 0 : (na < nb ? -1 : 1);
}
__device__ __forceinline__ bool diff_less(const DevBlock& b, u32 x, u32 y) {
    const tfbs_variant& vx = b.variants[x];
    const tfbs_variant& vy = b.variants[y];
    if (vx.pos != vy.pos) return vx.pos < vy.pos;
    int c = cmp_codes(b.allele_codes + vx.ref_off, vx.ref_len, b.allele_codes + vy.ref_off, vy.ref_len);
    if (c) return c < 0;
    return cmp_codes(b.allele_codes + vx.alt_off, vx.alt_len, b.allele_codes + vy.alt_off, vy.alt_len) < 0;
}

__device__ __forceinline__ void report(DevStatus* st, u64 q, i64 relpos, u32 code) {
    u64 key = (q << 32) | ((u64)((relpos + (1 << 27)) & 0xfffffff) << 4) | code;
    atomicMin(&st->err_key, key);
}

// patch_haplotype (haplotype.rs:98-153) over the sorted diff list dl[0, nd): the same cases in the same order, emitting segments
// instead of bases.  Returns the number of segments (the terminator is written behind them); st == NULL: panics are not
// reported (a configuration replays diffs whose haplotype has already reported them).
struct WalkOut {
    u32 ns, len, ntake;
    bool trunc;
    u32 err;  // DEV_* of the panic that ended the walk (reported to st only when st != NULL), else DEV_OK
};
template <class Sink>
__device__ __forceinline__ WalkOut walk_diffs_to(const DevBlock& b, u32 r, const u32* dl, u32 nd, Sink&& put, DevStatus* st, u64 q_report) {
    const i64 start = b.region_start[r], end = b.region_end[r];
    const u64 ro = b.ref_off[r];
    const i64 n_ref = (i64)(b.ref_off[r + 1] - ro);
    const i64 avail_end = start + n_ref - 1;
    u32 out = 0, ns = 0;
    bool trunc = false;
    u32 err = DEV_OK;
    i64 rp = start;
    auto emit_ref = [&](i64 a, i64 e2) {
        if (a < start) a = start;
        if (e2 > avail_end) e2 = avail_end;
        if (e2 >= a) {
            put(ns++, Seg{out, (u32)(a - start), (int)(a - start), 0u}, 0xffffffffu);
            out += (u32)(e2 - a + 1);
        }
    };
    u32 k = 0;
    for (;;) {
        if (k == nd) {  // haplotype.rs:100-108
            if (rp <= end) emit_ref(rp, end);
            break;
        }
        const tfbs_variant d = b.variants[dl[k]];
        if (d.pos > rp) {  // :110-114
            emit_ref(rp, d.pos - 1);
            rp = d.pos;
        } else if (d.pos == rp && d.ref_len == 1) {  // :115-135 SNV or insertion
            u8 at = (rp >= start && rp <= avail_end) ? b.ref_codes[ro + (u64)(rp - start)] : (u8)4;
            if (b.allele_codes[d.ref_off] != at) { err = DEV_REF_MISMATCH; if (st) report(st, q_report, rp - start, err); break; }
            put(ns++, Seg{out, d.alt_off, (int)(rp - start), 1u}, dl[k]);
            out += d.alt_len;
            rp += 1;
            ++k;
        } else if (d.pos == rp && d.alt_len == 1) {  // :136-140 deletion
            put(ns++, Seg{out, d.alt_off, (int)(rp - start), 1u}, dl[k]);
            out += 1;
            rp += d.ref_len;
            ++k;
        } else if (d.pos == rp) {  // :141-143
            err = DEV_MISSING_CASE;
            if (st) report(st, q_report, rp - start, err);
            break;
        } else if (rp >= end) {  // :144-146
            trunc = true;
            emit_ref(rp, rp);
            ++k;
            break;
        } else {  // :147-149
            trunc = true;
            ++k;
            break;
        }
    }
    put(ns, Seg{out, 0u, 0, 2u}, 0xffffffffu);  // terminator
    return WalkOut{ns, out, k, trunc, err};
}
__device__ __forceinline__ WalkOut walk_diffs(const DevBlock& b, u32 r, const u32* dl, u32 nd, Seg* sg, DevStatus* st, u64 q_report) {
    return walk_diffs_to(b, r, dl, nd, [sg](u32 i, const Seg& x, u32) { sg[i] = x; }, st, q_report);
}

// Thread per sequence: gathers the carried in-window diffs (haplotype.rs:95), sorts them (:96) and walks them.
// store_segs = 0: the segment lists are not kept (the configuration path scans virtual sequences, k_cfg_walk; only k_seq_resolve
// looks at a haplotype's own segments, for the few candidates of the sequence-keyed map, and walks those again).
__global__ void k_walk(DevBlock b, DevSeqs sq, u64 d_cap, DevStatus* st, u32 store_segs) {
    u32 q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= seq_count(sq)) return;
    u32 r = sq.seq_region[q];
    u32 h = sq.seq_leader[q];
    u64 doff = sq.seq_doff[q];
    if (doff + sq.seq_nd[q] > d_cap) return;  // the diff lists do not fit: the run is repeated with more scratch (need_d says how much)
    u32* dl = sq.dlist + doff;
    Seg* sg = sq.segs + 2 * doff + 2 * (u64)q;
    u32 nd = 0;
    auto take = [&](u32 v) {  // insertion sort; records come sorted by position, so this is nearly linear
        u32 k = nd++;
        while (k > 0 && diff_less(b, v, dl[k - 1])) { dl[k] = dl[k - 1]; --k; }
        dl[k] = v;
    };
    if (h != 0xffffffffu && b.hap_mask) {  // the set bits of the leader's mask
        const u32 v0 = b.var_off[r], nw = (b.var_off[r + 1] - v0 + 31) / 32;
        const u32* mask = b.hap_mask + b.mask_base[r] + h;
        for (u32 w = 0; w < nw; ++w)
            for (u32 m = mask[(u64)w * b.H]; m; m &= m - 1) {
                const u32 v = v0 + 32 * w + (u32)__ffs((int)m) - 1;
                if (b.var_inwin[v]) take(v);
            }
    } else if (h != 0xffffffffu) {
        for (u32 v = b.var_off[r]; v < b.var_off[r + 1]; ++v)
            if (b.var_inwin[v] && carries(b, v, h)) take(v);
    }
    // hash of the (nuc, pos) vector, segment by segment as the walk emits them (a segment's length is known when the next one starts)
    const u64* P = b.ref_prefix + b.ref_off[r] + r;
    u64 hsh = 0;
    Seg prev{0u, 0u, 0, 2u};
    u32 prev_v = 0xffffffffu;  // the record of an ALT segment: its bases' share of the hash is known per record (k_variant_prep)
    const WalkOut w = walk_diffs_to(b, r, dl, nd, [&](u32 i, const Seg& x, u32 v) {
        if (store_segs) sg[i] = x;
        if (i) {
            if (prev.kind == 0) {
                const u32 n = x.out_start - prev.out_start;
                hsh += hash_pow((long long)prev.out_start - (long long)prev.src) * (P[prev.src + n] - P[prev.src]);
            } else {
                hsh += hash_pow(prev.out_start) * b.var_althash[prev_v];
            }
        }
        prev = x;
        prev_v = v;
    }, st, q);
    sq.seq_nseg[q] = w.ns;
    sq.seq_len[q] = w.len;
    sq.seq_flags[q] = w.trunc ? 1 : 0;
    sq.seq_ntake[q] = w.ntake;
    sq.seq_hash[q] = hsh;
    if (w.trunc) atomicAdd(&st->n_truncated, 1u);
}

__device__ __forceinline__ u32 seg_find(const Seg* sg, u32 ns, u32 i) {  // last segment with out_start <= i
    u32 lo = 0, hi = ns;  // sg[ns] is the terminator
    while (hi - lo > 1) {
        u32 mid = (lo + hi) >> 1;
        if (sg[mid].out_start <= i) lo = mid; else hi = mid;
    }
    return lo;
}

// Prefix sums of val(code_t, t) * B^t over the window of every region (one CTA per region).
__global__ void k_ref_prefix(DevBlock b, u32 r0, u64* prefix) {
    __shared__ u64 s_carry;
    const u32 r = r0 + blockIdx.x;
    const u64 ro = b.ref_off[r];
    const u32 n = (u32)(b.ref_off[r + 1] - ro);
    u64* P = prefix + ro + r;
    if (threadIdx.x == 0) { s_carry = 0; P[0] = 0; }
    __syncthreads();
    for (u32 t0 = 0; t0 < n; t0 += SCAN_THREADS) {
        const u32 t = t0 + threadIdx.x;
        u64 term = t < n ? hash_val(b.ref_codes[ro + t], (int)t, b.hash_seed) * hash_pow(t) : 0ULL;
        u64 tot;
        u64 ex = block_exclusive_scan(term, &tot);
        const u64 carry = s_carry;
        if (t < n) P[t + 1] = carry + ex + term;
        __syncthreads();
        if (threadIdx.x == 0) s_carry = carry + tot;
        __syncthreads();
    }
}

__device__ __forceinline__ u32 seq_group(const DevSeqs& sq, u32 q) {  // group index of q inside its region (0 = the reference haplotype)
    if (sq.n_ref) return q < sq.n_ref ? 0u : 1u;  // virtual sequences: only "reference or not" is meaningful
    return (u32)((u64)q + sq.gbase0 - sq.gbase[sq.seq_region[q]]);
}

__global__ void k_seq_insert(DevSeqs sq, u64* keys, u32* vals, u32 mask, u32 seg, u32 r0) {  // seg, r0: see k_group_insert
    u32 q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= seq_count(sq)) return;
    u32 g = seq_group(sq, q);
    if (g == 0) return;  // the reference haplotype is not in the map (main.rs:129-147)
    u64 key = region_key(sq.seq_hash[q] + mix64(sq.seq_len[q]), sq.seq_region[q]);
    const u64 base = seg ? (u64)(sq.seq_region[q] - r0) * seg : 0;
    u32 slot = table_find_or_insert(keys + base, seg ? seg - 1 : mask, key);
    atomicMin(&vals[base + slot], g);
}

__device__ __forceinline__ void base_at(const DevBlock& b, const DevSeqs& sq, u32 q, u32 i, u8* c, int* rel) {
    const Seg* sg = sq.segs + 2 * sq.seq_doff[q] + 2 * (u64)q;
    u32 s = seg_find(sg, sq.seq_nseg[q], i);
    Seg cur = sg[s];
    u32 o = i - cur.out_start;
    if (cur.kind == 0) { *c = b.ref_codes[b.ref_off[sq.seq_region[q]] + cur.src + o]; *rel = cur.relpos + (int)o; }
    else { *c = b.allele_codes[cur.src + o]; *rel = cur.relpos; }
}

// A later insert with an equal key overwrites the earlier one in the reference (haplotype.rs:84); the
// winner there depends on HashMap order, here the group with the smallest first haplotype wins (same rule
// as the oracle).  The losers are dropped: their haplotypes stay in the reference set (main.rs:103-105).
__global__ void k_seq_resolve(DevBlock b, DevSeqs sq, const u64* keys, const u32* vals, u32 mask, u32 seg, u32 r0, DevStatus* st, u32 have_segs) {
    u32 q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= seq_count(sq)) return;
    u32 g = seq_group(sq, q);
    if (g == 0) return;
    u64 key = region_key(sq.seq_hash[q] + mix64(sq.seq_len[q]), sq.seq_region[q]);
    const u64 base = seg ? (u64)(sq.seq_region[q] - r0) * seg : 0;
    u32 slot = table_find(keys + base, seg ? seg - 1 : mask, key);
    u32 w = vals[base + slot];
    if (w == g) return;
    u32 qw = q - g + w;
    bool same = sq.seq_len[qw] == sq.seq_len[q] && sq.seq_region[qw] == sq.seq_region[q];
    // walk the two segment lists over the union of their breakpoints: two reference-copy pieces at the same position are equal by
    // construction, anything else is compared base by base (nuc and pos)
    if (same) {
        Seg* sa = sq.segs + 2 * sq.seq_doff[q] + 2 * (u64)q;
        Seg* sb = sq.segs + 2 * sq.seq_doff[qw] + 2 * (u64)qw;
        if (!have_segs) {  // k_walk did not keep them: walk the two candidates again into their own slots (several losers of one winner
                           // write the same values to the winner's slot)
            walk_diffs(b, sq.seq_region[q], sq.dlist + sq.seq_doff[q], sq.seq_nd[q], sa, nullptr, 0);
            walk_diffs(b, sq.seq_region[qw], sq.dlist + sq.seq_doff[qw], sq.seq_nd[qw], sb, nullptr, 0);
        }
        const u8* refc = b.ref_codes + b.ref_off[sq.seq_region[q]];
        const u32 len = sq.seq_len[q];
        u32 ia = 0, ib = 0, i = 0;
        while (same && i < len) {
            while (sa[ia + 1].out_start <= i) ++ia;
            while (sb[ib + 1].out_start <= i) ++ib;
            const u32 ea = sa[ia + 1].out_start, eb = sb[ib + 1].out_start;
            const u32 e = ea < eb ? ea : eb;
            const u32 da = i - sa[ia].out_start, db = i - sb[ib].out_start;
            if (sa[ia].kind == 0 && sb[ib].kind == 0) {
                same = sa[ia].relpos + (int)da == sb[ib].relpos + (int)db;
            } else {
                for (u32 x = 0; same && x < e - i; ++x) {
                    const u8 ca = sa[ia].kind == 0 ? refc[sa[ia].src + da + x] : b.allele_codes[sa[ia].src + da + x];
                    const u8 cb = sb[ib].kind == 0 ? refc[sb[ib].src + db + x] : b.allele_codes[sb[ib].src + db + x];
                    const int pa = sa[ia].relpos + (sa[ia].kind == 0 ? (int)(da + x) : 0);
                    const int pb = sb[ib].relpos + (sb[ib].kind == 0 ? (int)(db + x) : 0);
                    same = ca == cb && pa == pb;
                }
            }
            i = e;
        }
    }
    if (same) {
        sq.seq_flags[q] |= 2;
        atomicAdd(&st->n_dropped, 1u);
    } else {
        atomicAdd(&st->seq_collision, 1u);
    }
}

// cells a haplotype of `len` bases costs: sum over the patterns of max(0, len - L + 1) * L (pattern.rs:147-150)
__device__ __forceinline__ u64 cells_of_length(u32 len, u32 max_len, u32 sum_len, u64 sum_len_sq, u32 n_patterns, const u32* pat_len) {
    if (len >= max_len) return (u64)(len + 1) * sum_len - (sum_len_sq + sum_len);
    u64 cells = 0;
    for (u32 p = 0; p < n_patterns; ++p) {
        const u32 L = pat_len[p];
        if (L && len >= L) cells += (u64)(len - L + 1) * L;
    }
    return cells;
}

// hap_flags (audit only, else NULL): the flags of the haplotype's own diff list, taken before the redirect (TFBS_HAP_* bits).
// nominal (else NULL): the nominal cells -- every haplotype of every sample scanned on its own sequence (BASELINE.md "Unit of
// work") -- are added up here, in the pass that visits every haplotype anyway.
__global__ void k_redirect(u32 H, u32 r0, u32 nr, DevSeqs sq, u32* hap_group, u32* ref_used, u8* hap_flags, u64* nominal, u32 max_len,
                           u32 sum_len, u64 sum_len_sq, u32 n_patterns, const u32* pat_len) {
    u64 idx = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u64 cells = 0;
    if (idx < (u64)nr * H && !(sq.abort && *sq.abort)) {
        u32 r = r0 + (u32)(idx / H), h = (u32)(idx % H);
        u32 g = hap_group[(size_t)r * H + h];
        const u8 fl = g ? sq.seq_flags[sq.gbase[r] - sq.gbase0 + g] : (u8)0;
        if (hap_flags) hap_flags[(size_t)r * H + h] = fl;
        if (fl & 2) { g = 0; hap_group[(size_t)r * H + h] = 0; }
        if (g == 0) ref_used[r] = 1;
        if (nominal) cells = cells_of_length(sq.seq_len[sq.gbase[r] - sq.gbase0 + g], max_len, sum_len, sum_len_sq, n_patterns, pat_len);
    }
    if (nominal) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cells += __shfl_xor_sync(0xffffffffu, cells, o);
        if ((threadIdx.x & 31) == 0 && cells) atomicAdd((unsigned long long*)nominal, (unsigned long long)cells);
    }
}

}  // namespace tfbs
