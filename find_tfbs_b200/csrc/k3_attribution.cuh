// k3_attribution.cuh -- K3, configuration path, option "attribution": which configurations change each result row, and by how much
// Part of the sm_100a kernels of the find-tfbs hot path; included through kernels.cuh (see the map there).
//
// The fan-out (k3_fanout.cuh) builds a haplotype group's count for a key as C0[key] + the sum of D[key][c] over the group's live
// configurations c.  The launches here run right behind k_row_headers, while D, C0, the diff lists and the run arrays still belong to
// the block (the next block reuses them as scratch), and copy that sum's terms into per-slot result buffers (tfbs_attribution):
//   1. numbering: a configuration's output id is the block-wide rank of its representative diff-list entry (the smallest entry whose
//      run holds the same records).  Entries are laid out by (region, group, position), so the ids are ordered by region and do not
//      depend on hash seeds or on the atomic that numbered the difference matrix's columns (run_cfg).  A flag per entry, one scan.
//   2. per configuration its region, truncation flag and records; per distinct haplotype the output ids of its live runs (the runs
//      k_members files the group under), in diff-list order: a count, a scan, a fill.
//   3. terms: a warp per emitted row walks the region's configurations in output-id order and keeps the non-zero differences
//      (ballot + popc), once to count, once to fill behind a scan, so the order is fixed.
// The fan-out only reads D: the columns read here hold what the rows were built from.  The collect that returns the block copies the
// results to the host (fetch_attribution), so a later block in the same slot never races with a tfbs_get_attribution.
#pragma once
#include "k3_fanout.cuh"

namespace tfbs {

struct DevAttr {
    // scratch (shared by consecutive blocks)
    u32* e_flag;      // [d] 1 at the representative entry of a configuration
    u64* cfg_id;      // [d + 1] exclusive scan of e_flag: the output id at a representative entry
    u32* cfg_nrec;    // [cfg] records of the configuration (by output id)
    u32* cfg_col;     // [cfg] column of the configuration in its region's difference matrix
    u32* glist_n;     // [seq] live runs of the distinct haplotype
    u32* t_cnt;       // [rows] non-zero terms of the row
    // results (per slot)
    u32* cfg_region;  // [cfg]
    u8* cfg_flags;    // [cfg]
    u64* cfg_rec_off; // [cfg + 1]
    u32* cfg_rec;     // [d]
    u64* group_off;   // [seq + 1]
    u32* group_cfg;   // [d]
    u32* ref_count;   // [rows]
    u64* term_off;    // [rows + 1]
    u32* term_cfg;    // [terms]
    int* term_diff;   // [terms]
    u64 cfg_cap, d_cap, terms_cap;
};

__global__ void k_att_flags(DevConfigs cf, DevAttr at, const u64* n_d_ptr) {
    if (cf.plan->abort) return;
    const u64 n = *n_d_ptr < at.d_cap ? *n_d_ptr : at.d_cap;
    for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (u64)gridDim.x * blockDim.x)
        at.e_flag[e] = (cf.run_len[e] && cf.run_rep[e] == (u32)e) ? 1u : 0u;
}

// Thread per distinct haplotype: FILL = false describes the configurations it represents and counts its live runs; FILL = true copies
// the records of those configurations and lists the output ids of its live runs.
template <bool FILL>
__global__ void k_att_configs(DevSeqs sq, DevConfigs cf, DevSeqs vq, DevAttr at) {
    if (cf.plan->abort) return;
    const u32 q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= seq_count(sq)) return;
    const u64 doff = sq.seq_doff[q];
    const u32 nd = sq.seq_nd[q];
    if (doff + nd > at.d_cap) return;
    const u32 r = sq.seq_region[q];
    u32 live = 0;
    const u64 g0 = FILL ? at.group_off[q] : 0;
    for (u32 k = 0; k < nd; ++k) {
        const u64 e = doff + k;
        const u32 n = cf.run_len[e];
        if (!n) continue;
        if (FILL && g0 + live < at.d_cap) at.group_cfg[g0 + live] = (u32)at.cfg_id[cf.run_rep[e]];
        ++live;
        if (cf.run_rep[e] != (u32)e) continue;
        const u64 o = at.cfg_id[e];
        if (o >= at.cfg_cap) continue;
        if (FILL) {
            const u64 p = at.cfg_rec_off[o];
            for (u32 x = 0; x < n && p + x < at.d_cap; ++x) at.cfg_rec[p + x] = sq.dlist[e + x];
        } else {
            const u32 col = cf.run_cfg[e];
            at.cfg_region[o] = r;
            at.cfg_col[o] = col;
            at.cfg_nrec[o] = n;
            at.cfg_flags[o] = vq.seq_flags[(u64)vq.n_ref + cf.cfgbase[r] + col] & 1;
        }
    }
    if (!FILL) at.glist_n[q] = live;
}

// One CTA per region, a warp per key that became a row: the region's configurations in output-id order, the non-zero entries of the
// key's row of D.  FILL = false counts them (and writes the reference count), FILL = true writes them behind term_off.
template <bool FILL>
__global__ void k_att_terms(DevBlock b, DevConfigs cf, DevFan fn, DevAttr at, const u64* n_rows_ptr) {
    if (cf.plan->abort) return;
    const u32 r = blockIdx.x;
    const u32 lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const u32 nk = b.inner_off[r + 1] - b.inner_off[r];
    const u32 nkeys = fn.n_pid * nk;
    const u64 kb = cf.kbase[r];
    const u32 ncfg = cf.ncfg[r];
    const u64 o0 = cf.cfgbase[r];  // the region's output ids are [cfgbase[r], cfgbase[r] + ncfg): ids are ordered by region
    const u32* Dr = cf.D + cf.dbase[r];
    const u32 below = (1u << lane) - 1u;
    for (u32 key = wid; key < nkeys; key += nw) {
        if (!fn.flag[kb + key]) continue;
        const u64 row = fn.rowidx[kb + key];
        if (row >= fn.rows_cap || row >= *n_rows_ptr) continue;
        const u32* drow = Dr + (u64)key * ncfg;
        u64 t = FILL ? at.term_off[row] : 0;
        const u64 t_end = FILL ? at.term_off[row + 1] : 0;
        if (FILL && t_end > at.terms_cap) continue;  // the gate behind the count pass has raised abort
        u32 cnt = 0;
        for (u32 c0 = 0; c0 < ncfg; c0 += 32) {
            const u32 c = c0 + lane;
            const u32 d = c < ncfg ? drow[at.cfg_col[o0 + c]] : 0u;
            const u32 m = __ballot_sync(0xffffffffu, d != 0);
            if (FILL && d) {
                const u64 p = t + __popc(m & below);
                at.term_cfg[p] = (u32)(o0 + c);
                at.term_diff[p] = (int)d;
            }
            t += __popc(m);
            cnt += __popc(m);
        }
        if (!FILL && lane == 0) {
            at.t_cnt[row] = cnt;
            at.ref_count[row] = cf.C0[kb + key];
        }
    }
}

}  // namespace tfbs
