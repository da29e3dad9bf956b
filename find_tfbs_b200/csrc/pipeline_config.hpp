// pipeline_config.hpp -- the default path: configurations (k2c_configs.cuh), fan-out into grouped rows (k3_fanout.cuh), no host round trip
// Host side of libtfbs_b200.so (tfbs.cu is the map); one translation unit.
//
// enqueue() launches the whole pipeline of a block on the kernel stream of its lane and returns: every size that only the device
// learns (distinct haplotypes, carried records, configurations, work-list items, packed bases, rows) is met with a CAPACITY chosen
// from the previous blocks (tfbs_ctx::hint) and a gate kernel that publishes the real count; a count above its capacity raises
// DevPlan::abort, the later stages skip, and finalize() -- called from tfbs_collect, the only place the host waits -- repeats the
// block with the capacities the device asked for.  In steady state a block costs one wait.
#pragma once
#include "host_common.hpp"

namespace {

__global__ void k_status_init(DevStatus* st, DevPlan* plan) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        DevStatus s{};
        s.err_key = ~0ULL;
        s.bad_ref_base = ~0ULL;
        s.bad_allele_base = ~0ULL;
        *st = s;
        *plan = DevPlan{};
    }
}
__global__ void k_region_keys(DevBlock b, u32 n_pid, u32* nkeys) {
    const u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < b.R) nkeys[r] = n_pid * (b.inner_off[r + 1] - b.inner_off[r]);
}

// util.rs:15 / haplotype.rs:126-128,141-143: the reference's panics, as status codes with the same text
int patch_panic(tfbs_ctx* ctx, uint64_t err_key, uint32_t r, int64_t region_start) {
    int64_t rel = (int64_t)((err_key >> 4) & 0xfffffff) - (1 << 27);
    uint32_t code = (uint32_t)(err_key & 15);
    int64_t pos = region_start + rel;
    if (code == DEV_REF_MISMATCH)
        return fail(ctx, TFBS_ERR_REF_MISMATCH,
                    "First reference nucleotide of variant doesn't match reference genome: ref_position=" + std::to_string(pos) +
                        " region=" + std::to_string(r));
    return fail(ctx, TFBS_ERR_MISSING_CASE, "Missing case in haplotype patcher (ref_position=" + std::to_string(pos) + " region=" + std::to_string(r) + ")");
}

// groups a count vector of k_fanout<false> holds in dynamic shared memory next to the pairs and the staging buffer: the device's
// per-block limit less the kernel's static shared memory, at most 220 KB (53,120 groups on sm_100: 227 KB - 7.5 KB - 12 KB)
uint32_t fan_smem_groups(const cudaDeviceProp& prop) {
    return (uint32_t)((std::min<size_t>(prop.sharedMemPerBlockOptin - FAN_STATIC_SMEM, 220 * 1024) - fan_smem_bytes(0, 0, false)) / 4);
}

struct ConfigPipeline {
    tfbs_ctx* ctx;
    Slot* slot;
    Lane& L;  // the slot's streams and scratch
    BlockDev& B;
    cudaStream_t st;
    const uint32_t R, S, H;
    const uint64_t RH;
    uint32_t n_pid = 0;
    uint64_t n_keys = 0;
    DevStatus* dst = nullptr;
    DevPlan* plan = nullptr;
    DevBlock db{};
    uint64_t ref_items = 0;  // work-list items of the reference haplotypes (pieces of REF_PIECE window starts)
    const uint32_t smem_groups;  // fan_smem_groups()

    ConfigPipeline(tfbs_ctx* c, Slot* s)
        : ctx(c), slot(s), L(c->lane[s->lane]), B(*s->in), st(L.stream), R(s->in->R), S(s->in->S), H(s->in->H), RH((uint64_t)s->in->R * s->in->H),
          smem_groups(fan_smem_groups(c->prop)) {}

    uint32_t& launches() { return slot->stats.total_launches; }
    int scan(const uint32_t* d_in, uint64_t n_cap, const u64* n_ptr, u64* d_out) { return device_scan(ctx, L, d_in, n_cap, n_ptr, d_out, &launches()); }
    int gate(const u64* total, uint64_t add, uint64_t cap, u64* n_out, u64* need_out) {
        TFBS_LAUNCH(k_gate, 1, 1, 0, st)(total, (u64)add, (u64)cap, n_out, need_out, &plan->abort);
        ++launches();
        return TFBS_OK;
    }

    // ---- capacities ------------------------------------------------------------------------------------------------
    static uint64_t up(uint64_t need) { return need + need / 4 + 16; }
    // count vector for `need` groups: with the usual slack, but a need that fits shared memory is not pushed out of it by the slack
    uint32_t groups_for(uint64_t need) const {
        uint64_t cap = std::min<uint64_t>((uint64_t)H + 1, up(need));
        if (need <= smem_groups) cap = std::min<uint64_t>(cap, smem_groups);
        return (uint32_t)cap;
    }
    void choose_caps(bool first_attempt) {
        Caps& c = slot->caps;
        const Caps& h = ctx->hint;
        const uint64_t n_var = B.n_var;
        uint64_t ref_units = 0;
        ref_items = 0;
        for (uint32_t r = 0; r < R; ++r) {
            const uint64_t w = (uint64_t)(B.h_region_end[r] - B.h_region_start[r] + 1);
            const uint64_t pieces = w / REF_PIECE + 1;
            ref_items += pieces;
            ref_units += pieces * ((REF_PIECE + 64) / 32 + 2);
        }
        if (!first_attempt) return;  // a repeated run keeps the capacities finalize() grew
        if (ctx->tiny_caps) {  // testing: every growth path runs
            c = Caps{};
            c.seq = R; c.d = 1; c.cfg = 1; c.vd = 1; c.items = ref_items + 1; c.units = 1; c.dwords = 1; c.rows = 1; c.rowwords = 1; c.capr = 1; c.groups = 1; c.terms = 1;
            return;
        }
        // what the previous blocks needed (+ 25 %) when there is a history, else a guess from the shape of the block; a wrong guess
        // costs one repeated run of this block, never a wrong result
        auto pick = [](uint64_t hinted, uint64_t cold) { return hinted ? up(hinted) : cold; };
        c.seq = std::min<uint64_t>(RH + R, pick(h.seq, std::min<uint64_t>(RH + R, std::max<uint64_t>(R, ctx->scratch_bytes / 8 / 128))));
        c.seq = std::max<uint64_t>(c.seq, R);
        c.d = pick(h.d, std::min<uint64_t>(2 * c.seq, ctx->scratch_bytes / 4 / 72));
        c.cfg = pick(h.cfg, 4 * n_var + R);
        c.vd = pick(h.vd, 2 * c.cfg);
        c.items = ref_items + c.vd;  // the reference haplotypes in pieces, a configuration has at most one item per carried record
        c.units = std::max<uint64_t>(pick(h.units, 0), ref_units + 8 * c.cfg);
        c.dwords = pick(h.dwords, c.cfg * (n_keys / std::max<uint32_t>(1, R) + 1));
        c.rows = std::min<uint64_t>(std::max<uint64_t>(1, n_keys), pick(h.rows, std::max<uint64_t>(4096, n_keys / 4)));
        c.rowwords = pick(h.rowwords, c.rows * ((uint64_t)(H + 1) / 32 + 1));
        c.capr = ctx->refhit_cap_opt ? (uint32_t)std::max<int64_t>(1, ctx->refhit_cap_opt / std::max<uint32_t>(1, R)) : (uint32_t)pick(h.capr, 512);
        c.groups = h.groups ? groups_for(h.groups) : (uint32_t)std::min<uint64_t>((uint64_t)H + 1, 2048);
        c.terms = pick(h.terms, 4 * c.rows);
    }
    uint64_t scratch_bytes_needed() const {
        const Caps& c = slot->caps;
        uint64_t tbl = 1024, seg = 64;
        while (tbl < 2 * c.d) tbl <<= 1;
        while (seg < 2 * ((uint64_t)H + 1)) seg <<= 1;
        tbl = std::max<uint64_t>(tbl, (uint64_t)R * seg);
        return RH * 20 + tbl * 12 + c.seq * 50 + c.d * (4 + 32 + 20 + 4) + c.seq * 32 + c.cfg * 32 + (R + c.cfg) * 60 + c.vd * 36 + c.items * 28 +
               c.units * 12 + c.dwords * 4 + n_keys * 36 + (uint64_t)c.capr * R * sizeof(RefHit) + c.rows * 34 + c.rowwords * 4 + fan_vec_bytes() + attribution_bytes();
    }
    // option "attribution": scratch per diff-list entry, configuration, distinct haplotype and row, the per-slot results, the terms
    uint64_t attribution_bytes() const {
        const Caps& c = slot->caps;
        return ctx->attribution ? c.d * 20 + c.cfg * 21 + c.seq * 12 + c.rows * 16 + c.terms * 8 : 0;
    }

    // ---- fan-out: the count vectors in shared memory (k_fanout<false>, one CTA per unit) or in device memory (k_fanout<true>) ----
    // Device memory when a region may have more groups than shared memory holds, or when option fan_vector asks for it (testing).
    bool fan_vec() const { return ctx->fan_vector == 1 || slot->caps.groups > smem_groups; }
    // CTAs per region: FAN_SPLIT when there are many regions, more when few regions would leave SMs idle (sample blocks of a biobank
    // cohort: few regions, tens of thousands of groups each)
    uint32_t fan_split() const {
        return (uint32_t)std::min<uint64_t>(32, std::max<uint64_t>(FAN_SPLIT, (8ull * ctx->prop.multiProcessorCount + R - 1) / std::max<uint32_t>(1, R)));
    }
    uint32_t fan_vec_grid() const {
        return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)ctx->prop.multiProcessorCount * FAN_VEC_CTAS_PER_SM, (uint64_t)R * fan_split()));
    }
    uint64_t fan_vec_stride() const { return ((uint64_t)slot->caps.groups + 31) & ~31ull; }  // words of a CTA's slice, 128-byte aligned
    uint64_t fan_vec_bytes() const { return (n_keys && fan_vec()) ? (uint64_t)fan_vec_grid() * fan_vec_stride() * 4 : 0; }

    // ---- scratch -------------------------------------------------------------------------------------------------------
    int reserve() {
        const Caps& c = slot->caps;
        int rc;
#define RS(buf, bytes) if ((rc = grow(ctx, buf, std::max<uint64_t>(1, (uint64_t)(bytes))))) return rc
        if ((rc = reserve_encoding(ctx, L, B))) return rc;
        RS(slot->d_status, sizeof(DevStatus));
        RS(slot->d_plan, sizeof(DevPlan));
        RS(slot->d_hap_group, RH * 4);
        RS(slot->d_gbase, (uint64_t)(R + 1) * 8);
        RS(L.d_sig, RH * 8);
        RS(L.d_nd_in, RH * 4);
        RS(L.d_leader, RH * 4);
        RS(L.d_ngroups, (uint64_t)R * 4);
        RS(L.d_sum_nd, (uint64_t)R * 4);
        RS(L.d_ref_used, (uint64_t)R * 4);
        RS(L.d_kbase, (uint64_t)(R + 1) * 8);
        {
            uint64_t mask_words = 0;  // H * sum over the regions of ceil(V / 32)
            for (uint32_t r = 0; r < R; ++r) mask_words += (uint64_t)H * ((B.h_var_off[r + 1] - B.h_var_off[r] + 31) / 32);
            RS(L.d_hap_mask, mask_words * 4);
            RS(L.d_mask_base, (uint64_t)(R + 1) * 8);
            RS(L.d_region_dups, (uint64_t)R * 4);
            RS(L.d_var_row, B.n_var * 4);
        }
        RS(L.d_seq_region, c.seq * 4);
        RS(L.d_seq_leader, c.seq * 4);
        RS(L.d_seq_nd, c.seq * 4);
        RS(L.d_seq_doff, (c.seq + 1) * 8);
        RS(L.d_seq_nseg, c.seq * 4);
        RS(L.d_seq_len, c.seq * 4);
        RS(L.d_seq_hash, c.seq * 8);
        RS(L.d_seq_flags, c.seq);
        RS(L.d_seq_ntake, c.seq * 4);
        RS(L.d_dlist, c.d * 4);
        RS(L.d_segs, (2 * c.d + 2 * c.seq) * sizeof(Seg));
        RS(L.d_var_cluster, B.n_var * 4);
        RS(L.d_var_sorted, B.n_var * 4);
        RS(L.d_ncfg, (uint64_t)R * 4);
        RS(L.d_dwords, (uint64_t)R * 4);
        RS(L.d_cfgbase, (uint64_t)(R + 1) * 8);
        RS(L.d_dbase, (uint64_t)(R + 1) * 8);
        RS(L.d_run_len, c.d * 4);
        RS(L.d_run_key, c.d * 8);
        RS(L.d_run_rep, c.d * 4);
        RS(L.d_run_cfg, c.d * 4);
        RS(L.d_cfg_src, c.cfg * 4);
        RS(L.d_cfg_net, c.cfg * 4);
        RS(L.d_mcount, c.cfg * 4);
        RS(L.d_moff, (c.cfg + 1) * 8);
        RS(L.d_mfill, c.cfg * 4);
        RS(L.d_members, c.d * 4);
        const uint64_t nv = R + c.cfg;
        RS(L.d_vq_region, nv * 4);
        RS(L.d_vq_leader, nv * 4);
        RS(L.d_vq_nd, nv * 4);
        RS(L.d_vq_doff, (nv + 1) * 8);
        RS(L.d_vq_nseg, nv * 4);
        RS(L.d_vq_len, nv * 4);
        RS(L.d_vq_flags, nv);
        RS(L.d_vq_ntake, nv * 4);
        RS(L.d_vq_nitems, nv * 4);
        RS(L.d_vq_item_off, (nv + 1) * 8);
        RS(L.d_vq_dlist, c.vd * 4);
        RS(L.d_vq_segs, (2 * c.vd + 2 * nv) * sizeof(Seg));
        RS(L.d_items, c.items * sizeof(ScanItem));
        RS(L.d_list, c.items * 4);
        RS(L.d_ent_units, c.items * 4);
        RS(L.d_ent_uoff, (c.items + 1) * 8);
        RS(L.d_pk, c.units * 8);
        RS(L.d_nm, c.units * 4);
        RS(L.d_D, c.dwords * 4);
        RS(L.d_C0, n_keys * 4);
        RS(L.d_refhits, (uint64_t)c.capr * R * sizeof(RefHit));
        RS(L.d_refcnt, (uint64_t)R * 4);
        RS(L.d_vmin, n_keys * 4);
        RS(L.d_vmax, n_keys * 4);
        RS(L.d_flag, n_keys * 4);
        RS(L.d_rowwords, n_keys * 4);
        RS(L.d_kbits, n_keys);
        RS(L.d_rowidx, (n_keys + 1) * 8);
        RS(L.d_rowoff, (n_keys + 1) * 8);
        RS(slot->d_o_region, c.rows * 4);
        RS(slot->d_o_inner, c.rows * 4);
        RS(slot->d_o_pid, c.rows * 2);
        RS(slot->d_o_vmin, c.rows * 4);
        RS(slot->d_o_vmax, c.rows * 4);
        RS(slot->d_o_base, c.rows * 4);
        RS(slot->d_o_bits, c.rows);
        RS(slot->d_o_off, c.rows * 8);
        RS(slot->d_o_packed, c.rowwords * 4);
        if (fan_vec_bytes()) RS(L.d_fan_vec, fan_vec_bytes());
        if (ctx->attribution) {
            RS(L.d_att_eflag, c.d * 4);
            RS(L.d_att_cfgid, (c.d + 1) * 8);
            RS(L.d_att_nrec, c.cfg * 4);
            RS(L.d_att_col, c.cfg * 4);
            RS(L.d_att_gn, c.seq * 4);
            RS(L.d_att_tcnt, c.rows * 4);
            RS(slot->d_a_ref, c.rows * 4);
            RS(slot->d_a_toff, (c.rows + 1) * 8);
            RS(slot->d_a_tcfg, c.terms * 4);
            RS(slot->d_a_tdiff, c.terms * 4);
            RS(slot->d_a_creg, c.cfg * 4);
            RS(slot->d_a_cflags, c.cfg);
            RS(slot->d_a_croff, (c.cfg + 1) * 8);
            RS(slot->d_a_crec, c.d * 4);
            RS(slot->d_a_goff, (c.seq + 1) * 8);
            RS(slot->d_a_gcfg, c.d * 4);
        }
#undef RS
        CK(slot->h_status.reserve(sizeof(DevStatus), false));
        CK(slot->h_plan.reserve(sizeof(DevPlan), false));
        return TFBS_OK;
    }

    int table_slots(uint64_t slots) {  // the shared open-addressing table with room for `slots` slots, emptied
        int rc;
        if ((rc = grow(ctx, L.d_keys, slots * 8))) return rc;
        if ((rc = grow(ctx, L.d_vals, slots * 4))) return rc;
        CK(cudaMemsetAsync(L.d_keys.p, 0, slots * 8, st));
        CK(cudaMemsetAsync(L.d_vals.p, 0xff, slots * 4, st));
        return TFBS_OK;
    }
    int table(uint64_t entries, uint32_t* mask) {  // the same as one table of a power-of-two number of slots >= 2 * entries
        uint64_t cap = 1024;
        while (cap < 2 * entries) cap <<= 1;
        if (cap > (1ull << 31)) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "block too large for the grouping table: submit fewer regions at a time");
        int rc;
        if ((rc = grow(ctx, L.d_keys, cap * 8))) return rc;
        if ((rc = grow(ctx, L.d_vals, cap * 4))) return rc;
        CK(cudaMemsetAsync(L.d_keys.p, 0, cap * 8, st));
        CK(cudaMemsetAsync(L.d_vals.p, 0xff, cap * 4, st));
        *mask = (uint32_t)(cap - 1);
        return TFBS_OK;
    }

    // ---- the whole pipeline, enqueued ------------------------------------------------------------------------------------
    int enqueue(bool first_attempt) {
        int rc;
        const CompiledPatterns& cp = ctx->cp;
        n_pid = (uint32_t)cp.pid_list.size();
        n_keys = (uint64_t)n_pid * B.n_inner;
        slot->n_keys = n_keys;
        slot->rows_mode = ctx->rows_mode;
        slot->full_mode = false;
        if (first_attempt) {
            memset(&slot->stats, 0, sizeof slot->stats);
            slot->attempts = 0;
            slot->seed = 0x243f6a8885a308d3ull;
        }
        slot->stats.h2d_bytes = B.h2d_bytes;
        slot->stats.sm_count = (uint32_t)ctx->prop.multiProcessorCount;
        slot->stats.total_launches = 0;
        slot->stats.scan_launches = 0;
        slot->stats.scan_input_bytes = 0;
        slot->res.n_rows = 0;
        slot->res.have_dense = slot->res.have_grouped = slot->res.have_attribution = false;
        slot->attribution = ctx->attribution != 0;
        choose_caps(first_attempt);
        const Caps& c = slot->caps;
        const bool fans = n_keys && R && S;
        slot->fan_groups_cap = fans ? c.groups : 0;
        slot->fan_ctas = fans ? (fan_vec() ? fan_vec_grid() : (uint32_t)std::min<uint64_t>(0xffffffffu, (uint64_t)R * fan_split())) : 0;
        slot->fan_in_device_memory = (fans && fan_vec()) ? 1 : 0;
        if (fan_vec_bytes() > ctx->scratch_bytes)
            return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "the fan-out's count vectors for " + std::to_string(c.groups) + " distinct haplotypes per region need about " +
                                                            std::to_string(fan_vec_bytes() >> 20) + " MB of device scratch, option scratch_mb allows " +
                                                            std::to_string(ctx->scratch_bytes >> 20));
        if (scratch_bytes_needed() > ctx->scratch_bytes)
            return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "the block needs about " + std::to_string(scratch_bytes_needed() >> 20) +
                                                            " MB of device scratch, option scratch_mb allows " + std::to_string(ctx->scratch_bytes >> 20) +
                                                            ": submit fewer regions per block");
        if (c.seq > 0x7fffffffull || c.d > 0xfffffff0ull || R + c.cfg > 0x7fffffffull || c.items > 0xfffffff0ull ||
            (fan_vec() && (uint64_t)R * fan_split() > 0xffffffffull))
            return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "block too large for 32-bit work-list indices: submit fewer regions per block");
        if ((rc = reserve())) return rc;
        dst = slot->d_status.as<DevStatus>();
        plan = slot->d_plan.as<DevPlan>();
        CK(cudaStreamWaitEvent(st, slot->ev_in, 0));  // the block's host -> device copies (stream_in)
        CK(cudaEventRecord(slot->ev_t[0], st));
        TFBS_LAUNCH(k_status_init, 1, 32, 0, st)(dst, plan);
        ++launches();
        if (R == 0 || S == 0) return finish_enqueue();

        // ---- inputs: ASCII -> codes, Diff classes, prefix hashes of the reference windows, keys per region ----
        const unsigned enc_grid = slot->stats.sm_count * 16;
        if (B.n_ref_bytes) {
            TFBS_LAUNCH(k_encode, std::min<unsigned>(grid_for(B.n_ref_bytes, 256), enc_grid), 256, 0, st)(B.d_ref_ascii.as<u8>(), L.d_ref_codes.as<u8>(), B.n_ref_bytes, &dst->bad_ref_base);
            ++launches();
        }
        if (B.n_allele_bytes) {
            TFBS_LAUNCH(k_encode, std::min<unsigned>(grid_for(B.n_allele_bytes, 256), enc_grid), 256, 0, st)(B.d_allele_ascii.as<u8>(), L.d_allele_codes.as<u8>(), B.n_allele_bytes, &dst->bad_allele_base);
            ++launches();
        }
        db = dev_block(L, B);
        db.hap_mask = L.d_hap_mask.as<u32>();
        db.mask_base = L.d_mask_base.as<u64>();
        db.region_dups = L.d_region_dups.as<u32>();
        db.var_row = db.var_row_out = L.d_var_row.as<u32>();
        db.hash_seed = slot->seed;
        TFBS_LAUNCH(k_mask_words, grid_for(R, 256), 256, 0, st)(db, L.d_dwords.as<u32>());
        ++launches();
        if ((rc = scan(L.d_dwords.as<u32>(), R, nullptr, L.d_mask_base.as<u64>()))) return rc;
        TFBS_LAUNCH(k_variant_prep, R, 128, 0, st)(db, 0, L.d_var_class.as<u32>(), L.d_var_inwin.as<u8>(), L.d_region_dups.as<u32>());
        TFBS_LAUNCH(k_ref_prefix, R, SCAN_THREADS, 0, st)(db, 0, L.d_ref_prefix.as<u64>());
        TFBS_LAUNCH(k_region_keys, grid_for(R, 256), 256, 0, st)(db, n_pid, L.d_dwords.as<u32>());
        launches() += 3;
        if ((rc = scan(L.d_dwords.as<u32>(), R, nullptr, L.d_kbase.as<u64>()))) return rc;

        // ---- K0: grouping by Vec<Diff> (haplotype.rs:65-75) ----
        u32* hap_group = slot->d_hap_group.as<u32>();
        // the tables of K0 and of the sequence-keyed map: one segment of `seg` slots per region (L2-resident while the region is worked on)
        uint32_t seg = 64;
        while (seg < 2 * ((uint64_t)H + 1)) seg <<= 1;
        {
            const uint64_t max_pairs = 1ull << 25;
            const uint32_t regions_per_super = (uint32_t)std::max<uint64_t>(1, max_pairs / std::max<uint32_t>(1, H));
            for (uint32_t r0 = 0; r0 < R; r0 += regions_per_super) {
                const uint32_t nr = std::min(regions_per_super, R - r0);
                const uint64_t pairs = (uint64_t)nr * H;
                if ((rc = table_slots((uint64_t)nr * seg))) return rc;
                TFBS_LAUNCH(k_signatures, grid_for((uint64_t)nr * ((H + 31) / 32) * 32, 256), 256, 0, st)(db, r0, nr, slot->seed, L.d_sig.as<u64>(), L.d_nd_in.as<u32>());
                TFBS_LAUNCH(k_group_insert, grid_for(pairs, 256), 256, 0, st)(H, r0, nr, L.d_sig.as<u64>(), L.d_keys.as<u64>(), L.d_vals.as<u32>(), 0u, seg);
                TFBS_LAUNCH(k_group_lookup, grid_for(pairs, 256), 256, 0, st)(db, r0, nr, L.d_sig.as<u64>(), L.d_keys.as<u64>(), L.d_vals.as<u32>(), 0u, seg,
                                                                     L.d_leader.as<u32>(), dst);
                TFBS_LAUNCH(k_group_rank, nr, 256, 0, st)(H, r0, L.d_leader.as<u32>(), L.d_nd_in.as<u32>(), hap_group, L.d_ngroups.as<u32>(),
                                                 L.d_sum_nd.as<u32>());
                launches() += 4;
            }
        }
        u64* gbase = slot->d_gbase.as<u64>();
        if ((rc = scan(L.d_ngroups.as<u32>(), R, nullptr, gbase))) return rc;
        gate(gbase + R, 0, c.seq, &plan->n_seq, &plan->need_seq);
        CK(cudaEventRecord(slot->ev_t[1], st));

        // ---- K1: patch_haplotype per distinct haplotype (segments + hash), the sequence-keyed map (haplotype.rs:81-85) ----
        DevSeqs sq{};
        sq.n_seq = (u32)c.seq;
        sq.n_seq_ptr = &plan->n_seq;
        sq.abort = &plan->abort;
        sq.gbase = gbase;
        sq.gbase0 = 0;
        sq.seq_region = L.d_seq_region.as<u32>();
        sq.seq_leader = L.d_seq_leader.as<u32>();
        sq.seq_nd = L.d_seq_nd.as<u32>();
        sq.seq_doff = L.d_seq_doff.as<u64>();
        sq.dlist = L.d_dlist.as<u32>();
        sq.segs = L.d_segs.as<Seg>();
        sq.seq_nseg = L.d_seq_nseg.as<u32>();
        sq.seq_len = L.d_seq_len.as<u32>();
        sq.seq_hash = L.d_seq_hash.as<u64>();
        sq.seq_flags = L.d_seq_flags.as<u8>();
        sq.seq_ntake = L.d_seq_ntake.as<u32>();
        TFBS_LAUNCH(k_seq_init, R, 128, 0, st)(H, 0, hap_group, L.d_leader.as<u32>(), L.d_nd_in.as<u32>(), sq);
        ++launches();
        if ((rc = scan(sq.seq_nd, c.seq, &plan->n_seq, sq.seq_doff))) return rc;
        // the total sits behind the last sequence; k_gate reads it through the clamped count
        TFBS_LAUNCH(k_gate_at, 1, 1, 0, st)(sq.seq_doff, &plan->n_seq, (u64)c.d, &plan->n_d, &plan->need_d, &plan->abort);
        ++launches();
        TFBS_LAUNCH(k_walk, grid_for(c.seq, 128), 128, 0, st)(db, sq, (u64)c.d, dst, 0u);
        ++launches();
        {
            if ((rc = table_slots((uint64_t)R * seg))) return rc;  // at most H + 1 distinct haplotypes per region
            CK(cudaMemsetAsync(L.d_ref_used.p, 0, (size_t)R * 4, st));
            TFBS_LAUNCH(k_seq_insert, grid_for(c.seq, 256), 256, 0, st)(sq, L.d_keys.as<u64>(), L.d_vals.as<u32>(), 0u, seg, 0u);
            TFBS_LAUNCH(k_seq_resolve, grid_for(c.seq, 128), 128, 0, st)(db, sq, L.d_keys.as<u64>(), L.d_vals.as<u32>(), 0u, seg, 0u, dst, 0u);
            TFBS_LAUNCH(k_redirect, grid_for(RH, 256), 256, 0, st)(H, 0, R, sq, hap_group, L.d_ref_used.as<u32>(), (u8*)nullptr, (u64*)&dst->nominal_cells,
                                                                   ctx->dpat.max_len, ctx->dpat.sum_len, (u64)ctx->dpat.sum_len_sq, ctx->dpat.n_patterns, ctx->dpat.pat_len);
            launches() += 3;
        }
        CK(cudaEventRecord(slot->ev_t[2], st));

        // ---- configurations ----
        DevConfigs cf{};
        cf.max_len = cp.max_len;
        cf.n_pid = n_pid;
        cf.var_cluster = L.d_var_cluster.as<u32>();
        cf.var_sorted = L.d_var_sorted.as<u32>();
        cf.ncfg = L.d_ncfg.as<u32>();
        cf.cfgbase = L.d_cfgbase.as<u64>();
        cf.dwords = L.d_dwords.as<u32>();
        cf.dbase = L.d_dbase.as<u64>();
        cf.kbase = L.d_kbase.as<u64>();
        cf.run_len = L.d_run_len.as<u32>();
        cf.run_key = L.d_run_key.as<u64>();
        cf.run_rep = L.d_run_rep.as<u32>();
        cf.run_cfg = L.d_run_cfg.as<u32>();
        cf.cfg_src = L.d_cfg_src.as<u32>();
        cf.cfg_net = L.d_cfg_net.as<int>();
        cf.mcount = L.d_mcount.as<u32>();
        cf.moff = L.d_moff.as<u64>();
        cf.mfill = L.d_mfill.as<u32>();
        cf.members = L.d_members.as<u32>();
        cf.D = L.d_D.as<u32>();
        cf.C0 = L.d_C0.as<u32>();
        cf.plan = plan;
        TFBS_LAUNCH(k_cluster, R, 128, 0, st)(db, cf);
        ++launches();
        {
            uint32_t mask;
            if ((rc = table(c.d, &mask))) return rc;
            CK(cudaMemsetAsync(cf.ncfg, 0, (size_t)R * 4, st));
            TFBS_LAUNCH(k_cfg_runs, grid_for(c.seq, 128), 128, 0, st)(db, sq, cf, (u64)c.d, slot->seed, L.d_keys.as<u64>(), L.d_vals.as<u32>(), mask);
            TFBS_LAUNCH(k_cfg_resolve, grid_for(c.seq, 128), 128, 0, st)(sq, cf, (u64)c.d, L.d_keys.as<u64>(), L.d_vals.as<u32>(), mask);
            launches() += 2;
        }
        TFBS_LAUNCH(k_region_sizes, grid_for(R, 256), 256, 0, st)(db, cf);
        ++launches();
        if ((rc = scan(cf.ncfg, R, nullptr, cf.cfgbase))) return rc;
        if ((rc = scan(cf.dwords, R, nullptr, cf.dbase))) return rc;
        gate(cf.cfgbase + R, 0, c.cfg, &plan->n_cfg, &plan->need_cfg);
        gate(cf.cfgbase + R, R, R + c.cfg, &plan->n_vseq, &plan->unused);
        gate(cf.dbase + R, 0, c.dwords, &plan->n_dwords, &plan->need_dwords);

        // virtual sequences: the reference haplotype of every region, then the configurations
        DevSeqs vq{};
        vq.n_seq = (u32)(R + c.cfg);
        vq.n_seq_ptr = &plan->n_vseq;
        vq.abort = &plan->abort;
        vq.n_ref = R;
        vq.seq_region = L.d_vq_region.as<u32>();
        vq.seq_leader = L.d_vq_leader.as<u32>();
        vq.seq_nd = L.d_vq_nd.as<u32>();
        vq.seq_doff = L.d_vq_doff.as<u64>();
        vq.dlist = L.d_vq_dlist.as<u32>();
        vq.segs = L.d_vq_segs.as<Seg>();
        vq.seq_nseg = L.d_vq_nseg.as<u32>();
        vq.seq_len = L.d_vq_len.as<u32>();
        vq.seq_flags = L.d_vq_flags.as<u8>();
        vq.seq_ntake = L.d_vq_ntake.as<u32>();
        vq.seq_nitems = L.d_vq_nitems.as<u32>();
        vq.item_off = L.d_vq_item_off.as<u64>();
        vq.items = L.d_items.as<ScanItem>();
        vq.n_items_cap = (u32)c.items;
        vq.ent_units = L.d_ent_units.as<u32>();
        vq.ent_uoff = L.d_ent_uoff.as<u64>();
        vq.pk = L.d_pk.as<u64>();
        vq.nm = L.d_nm.as<u32>();
        vq.units_cap = c.units;
        TFBS_LAUNCH(k_vseq_init, grid_for(R, 256), 256, 0, st)(R, vq);
        TFBS_LAUNCH(k_cfg_fill, grid_for(c.seq, 128), 128, 0, st)(sq, cf, vq, (u64)c.d);
        launches() += 2;
        if ((rc = scan(vq.seq_nd, R + c.cfg, &plan->n_vseq, vq.seq_doff))) return rc;
        TFBS_LAUNCH(k_gate_at, 1, 1, 0, st)(vq.seq_doff, &plan->n_vseq, (u64)c.vd, &plan->n_vd, &plan->need_vd, &plan->abort);
        ++launches();
        TFBS_LAUNCH(k_cfg_walk, grid_for(R + c.cfg, 128), 128, 0, st)(db, sq, cf, vq, (u64)c.vd);
        ++launches();

        // ---- work list, packed bases ----
        TFBS_LAUNCH(k_vitems<false>, grid_for(R + c.cfg, 128), 128, 0, st)(vq, cp.max_len, &plan->abort);
        ++launches();
        if ((rc = scan(vq.seq_nitems, R + c.cfg, &plan->n_vseq, vq.item_off))) return rc;
        TFBS_LAUNCH(k_gate_at, 1, 1, 0, st)(vq.item_off, &plan->n_vseq, (u64)c.items, &plan->n_items, &plan->need_items, &plan->abort);
        TFBS_LAUNCH(k_vitems<true>, grid_for(R + c.cfg, 128), 128, 0, st)(vq, cp.max_len, &plan->abort);
        TFBS_LAUNCH(k_vitem_units, grid_for(c.items, 256), 256, 0, st)(vq, &plan->n_items, L.d_list.as<u32>());
        launches() += 3;
        if ((rc = scan(vq.ent_units, c.items, &plan->n_items, vq.ent_uoff))) return rc;
        TFBS_LAUNCH(k_gate_at, 1, 1, 0, st)(vq.ent_uoff, &plan->n_items, (u64)c.units, &plan->n_units, &plan->need_units, &plan->abort);
        TFBS_LAUNCH(k_emit_list, grid_for(c.items * EMIT_LANES, 256), 256, 0, st)(db, vq, L.d_list.as<u32>(), &plan->n_items);
        TFBS_LAUNCH(k_item_stats, grid_for(c.items, 256), 256, 0, st)(vq, ctx->dpat, L.d_list.as<u32>(), &plan->n_items, dst);
        launches() += 3;

        // ---- the scan: one launch per pattern chunk ----
        TFBS_LAUNCH(k_zero_words, slot->stats.sm_count * 8, 256, 0, st)(cf.D, &plan->n_dwords, (u64)c.dwords);
        ++launches();
        if (n_keys) CK(cudaMemsetAsync(cf.C0, 0, n_keys * 4, st));
        CK(cudaMemsetAsync(L.d_refcnt.p, 0, (size_t)R * 4, st));
        DevRefHits drh{L.d_refhits.as<RefHit>(), L.d_refcnt.as<u32>(), c.capr, 0};
        DevCounts dc{cf.C0, cf.kbase, 0};
        DevMatches dm{};
        const int smem_bytes = (int)(sizeof(CtaShared) + SCAN_WARPS * sizeof(WarpShared) + ((cp.max_chunk_bytes + 15) & ~15u));
        const bool wide = cp.fields == 2;
        if (wide) CK(cudaFuncSetAttribute(k_scan<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
        else CK(cudaFuncSetAttribute(k_scan<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
        uint32_t scan_grid = (uint32_t)ctx->prop.multiProcessorCount;  // persistent: one CTA per SM shares one copy of the tables
        if (ctx->scan_ctas_per_sm < 0) scan_grid = (uint32_t)std::max(1, -ctx->scan_ctas_per_sm);
        slot->stats.scan_ctas = scan_grid;
        CK(cudaEventRecord(slot->ev_t[3], st));
        for (uint32_t ch = 0; ch < cp.chunks.size(); ++ch) {
            CK(cudaMemsetAsync(&dst->work_counter, 0, 4, st));
            if (wide) TFBS_LAUNCH(k_scan<2>, scan_grid, SCAN_CTA, smem_bytes, st)(db, vq, ctx->dpat, dc, dm, drh, cf, 1, L.d_list.as<u32>(), &plan->n_items, (u32)SCAN_PER_GRAB, dst, ch);
            else TFBS_LAUNCH(k_scan<3>, scan_grid, SCAN_CTA, smem_bytes, st)(db, vq, ctx->dpat, dc, dm, drh, cf, 1, L.d_list.as<u32>(), &plan->n_items, (u32)SCAN_PER_GRAB, dst, ch);
            ++launches();
            ++slot->stats.scan_launches;
        }
        CK(cudaEventRecord(slot->ev_t[4], st));

        // ---- lost reference hits, members of the configurations, counters ----
        TFBS_LAUNCH(k_refhit_need, grid_for(R, 256), 256, 0, st)(drh, R, plan);
        TFBS_LAUNCH(k_cfg_lost, grid_for(c.cfg * 8, 256), 256, 0, st)(db, vq, cf, drh);
        launches() += 2;
        CK(cudaMemsetAsync(cf.mcount, 0, c.cfg * 4, st));
        CK(cudaMemsetAsync(cf.mfill, 0, c.cfg * 4, st));
        TFBS_LAUNCH(k_members<false>, grid_for(c.seq, 128), 128, 0, st)(sq, cf, drh, L.d_ref_used.as<u32>(), (u64)c.d, ctx->dpat, dst);
        ++launches();
        if ((rc = scan(cf.mcount, c.cfg, &plan->n_cfg, cf.moff))) return rc;
        TFBS_LAUNCH(k_gate_at, 1, 1, 0, st)(cf.moff, &plan->n_cfg, (u64)c.d, &plan->n_members, &plan->need_members, &plan->abort);
        TFBS_LAUNCH(k_members<true>, grid_for(c.seq, 128), 128, 0, st)(sq, cf, drh, L.d_ref_used.as<u32>(), (u64)c.d, ctx->dpat, dst);
        launches() += 2;
        CK(cudaEventRecord(slot->ev_t[5], st));

        // ---- K3: fan-out, min / max filter, grouped rows ----
        if (n_keys) {
            DevFan fn{};
            fn.hap_group = hap_group;
            fn.gbase = gbase;
            fn.n_pid = n_pid;
            fn.rows_mode = ctx->rows_mode;
            fn.groups_cap = c.groups;
            fn.vmin = L.d_vmin.as<u32>();
            fn.vmax = L.d_vmax.as<u32>();
            fn.flag = L.d_flag.as<u32>();
            fn.k_base = L.d_rowwords.as<u32>();
            fn.k_bits = L.d_kbits.as<u8>();
            fn.k_off = L.d_rowoff.as<u64>();
            fn.rowidx = L.d_rowidx.as<u64>();
            fn.rows_cap = c.rows;
            fn.words_cap = c.rowwords;
            fn.o_region = slot->d_o_region.as<u32>();
            fn.o_inner = slot->d_o_inner.as<u32>();
            fn.o_pid = slot->d_o_pid.as<u16>();
            fn.o_vmin = slot->d_o_vmin.as<u32>();
            fn.o_vmax = slot->d_o_vmax.as<u32>();
            fn.o_base = slot->d_o_base.as<u32>();
            fn.o_bits = slot->d_o_bits.as<u8>();
            fn.o_off = slot->d_o_off.as<u64>();
            fn.o_packed = slot->d_o_packed.as<u32>();
            fn.pid_list = ctx->d_pid_list.as<u16>();
            fn.max_count = &dst->max_count;
            // shared memory: the pairs of a round, the staged rows, (when it fits) the haplotype -> group map and, unless the count
            // vectors are in device memory, one count vector per CTA (c.groups <= smem_groups there)
            const bool vec = fan_vec();
            const uint32_t smem_vec_groups = vec ? 0u : c.groups;
            fn.hg16 = ((uint64_t)H + 1 <= 65536 && fan_smem_bytes(smem_vec_groups, H, true) <= 64 * 1024) ? 1u : 0u;
            const size_t fan_smem = fan_smem_bytes(smem_vec_groups, H, fn.hg16 != 0);
            const uint32_t split = fan_split();
            if (vec) {
                fn.vec = L.d_fan_vec.as<u32>();
                fn.vec_stride = fan_vec_stride();
                fn.split = split;
                // the kernel leaves every slice all zero, a fresh or regrown allocation is not: zeroed on every run, repeats included
                CK(cudaMemsetAsync(L.d_fan_vec.p, 0, fan_vec_bytes(), st));
                CK(cudaFuncSetAttribute(k_fanout<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fan_smem));
                TFBS_LAUNCH(k_fanout<true>, fan_vec_grid(), FAN_THREADS, fan_smem, st)(db, cf, fn);
            } else {
                CK(cudaFuncSetAttribute(k_fanout<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fan_smem));
                CK(cudaFuncSetAttribute(k_fanout<false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
                TFBS_LAUNCH(k_fanout<false>, dim3(R, split), FAN_THREADS, fan_smem, st)(db, cf, fn);
            }
            ++launches();
            if ((rc = scan(fn.flag, n_keys, nullptr, L.d_rowidx.as<u64>()))) return rc;
            gate(L.d_rowidx.as<u64>() + n_keys, 0, c.rows, &plan->n_rows, &plan->need_rows);
            gate(&plan->rowwords_alloc, 0, c.rowwords, &plan->n_rowwords, &plan->need_rowwords);
            TFBS_LAUNCH(k_row_headers, R, 128, 0, st)(db, cf, fn, &plan->n_rows);
            ++launches();
            if (ctx->attribution && (rc = enqueue_attribution(sq, cf, vq, &fn))) return rc;
        } else if (ctx->attribution && (rc = enqueue_attribution(sq, cf, vq, nullptr))) {
            return rc;
        }
        return finish_enqueue();
    }

    // ---- option "attribution" (k3_attribution.cuh): behind the row headers, while D, C0, the diff lists and the runs are this block's ----
    // 6 launches, 4 more for the terms when the block has keys
    int enqueue_attribution(const DevSeqs& sq, const DevConfigs& cf, const DevSeqs& vq, const DevFan* fn) {
        const Caps& c = slot->caps;
        int rc;
        DevAttr at{};
        at.e_flag = L.d_att_eflag.as<u32>();
        at.cfg_id = L.d_att_cfgid.as<u64>();
        at.cfg_nrec = L.d_att_nrec.as<u32>();
        at.cfg_col = L.d_att_col.as<u32>();
        at.glist_n = L.d_att_gn.as<u32>();
        at.t_cnt = L.d_att_tcnt.as<u32>();
        at.cfg_region = slot->d_a_creg.as<u32>();
        at.cfg_flags = slot->d_a_cflags.as<u8>();
        at.cfg_rec_off = slot->d_a_croff.as<u64>();
        at.cfg_rec = slot->d_a_crec.as<u32>();
        at.group_off = slot->d_a_goff.as<u64>();
        at.group_cfg = slot->d_a_gcfg.as<u32>();
        at.ref_count = slot->d_a_ref.as<u32>();
        at.term_off = slot->d_a_toff.as<u64>();
        at.term_cfg = slot->d_a_tcfg.as<u32>();
        at.term_diff = slot->d_a_tdiff.as<int>();
        at.cfg_cap = c.cfg;
        at.d_cap = c.d;
        at.terms_cap = c.terms;
        // 1. output ids: the rank of the representative entries in diff-list order
        TFBS_LAUNCH(k_att_flags, slot->stats.sm_count * 8, 256, 0, st)(cf, at, &plan->n_d);
        ++launches();
        if ((rc = scan(at.e_flag, c.d, &plan->n_d, at.cfg_id))) return rc;
        // 2. configurations and group lists: describe + count, two scans, fill
        TFBS_LAUNCH(k_att_configs<false>, grid_for(c.seq, 128), 128, 0, st)(sq, cf, vq, at);
        ++launches();
        if ((rc = scan(at.cfg_nrec, c.cfg, &plan->n_cfg, at.cfg_rec_off))) return rc;
        if ((rc = scan(at.glist_n, c.seq, &plan->n_seq, at.group_off))) return rc;
        TFBS_LAUNCH(k_att_configs<true>, grid_for(c.seq, 128), 128, 0, st)(sq, cf, vq, at);
        ++launches();
        if (!fn) return TFBS_OK;
        // 3. terms: count, scan, gate, fill
        TFBS_LAUNCH(k_att_terms<false>, R, 256, 0, st)(db, cf, *fn, at, &plan->n_rows);
        ++launches();
        if ((rc = scan(at.t_cnt, c.rows, &plan->n_rows, at.term_off))) return rc;
        TFBS_LAUNCH(k_gate_at, 1, 1, 0, st)(at.term_off, &plan->n_rows, (u64)c.terms, &plan->n_terms, &plan->need_terms, &plan->abort);
        TFBS_LAUNCH(k_att_terms<true>, R, 256, 0, st)(db, cf, *fn, at, &plan->n_rows);
        launches() += 2;
        return TFBS_OK;
    }

    int finish_enqueue() {
        CK(cudaEventRecord(slot->ev_t[6], st));
        CK(cudaMemcpyAsync(slot->h_status.p, dst, sizeof(DevStatus), cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(slot->h_plan.p, plan, sizeof(DevPlan), cudaMemcpyDeviceToHost, st));
        CK(cudaEventRecord(slot->ev_done, st));
        CK(cudaGetLastError());
        slot->state = 1;
        return TFBS_OK;
    }

    // ---- tfbs_collect: wait, repeat with more scratch if the device asked for it, fetch the rows ----------------------------
    int finalize() {
        for (;;) {
            CK(cudaEventSynchronize(slot->ev_done));
            DevStatus hs;
            DevPlan hp;
            memcpy(&hs, slot->h_status.p, sizeof hs);
            memcpy(&hp, slot->h_plan.p, sizeof hp);
            if (hs.bad_ref_base != ~0ull || hs.bad_allele_base != ~0ull) {
                // util.rs:15 panic!("Unknown nucleotide {}", l)
                return fail(ctx, TFBS_ERR_UNKNOWN_NUCLEOTIDE,
                            std::string("Unknown nucleotide at byte ") + std::to_string(hs.bad_ref_base != ~0ull ? hs.bad_ref_base : hs.bad_allele_base) +
                                (hs.bad_ref_base != ~0ull ? " of ref_bases" : " of allele_bases"));
            }
            const bool collided = (hs.sig_collision && ctx->verify_groups) || hp.cfg_collision || hs.seq_collision ||  // every hash is seeded by slot->seed
                                  (ctx->test_reseed && slot->attempts == 0 && !hp.abort);
            if (!hp.abort && !collided) {
                if (hs.err_key != ~0ull) {
                    // region of sequence q: the status word carries the sequence; its region comes from the device's gbase
                    const uint32_t q = (uint32_t)(hs.err_key >> 32);
                    std::vector<uint64_t> gb(R + 1);
                    CK(cudaMemcpyAsync(gb.data(), slot->d_gbase.p, (size_t)(R + 1) * 8, cudaMemcpyDeviceToHost, st));
                    CK(cudaStreamSynchronize(st));
                    const uint32_t r = (uint32_t)(std::upper_bound(gb.begin(), gb.begin() + R, (uint64_t)q) - gb.begin() - 1);
                    return patch_panic(ctx, hs.err_key, r, B.h_region_start[r]);
                }
                note_needs(hp);
                return publish(hs, hp);
            }
            // repeat the block: a hash collision with another seed, an overflow with the capacities the device asked for
            if (++slot->attempts > 16) return fail(ctx, TFBS_ERR_INTERNAL, "the block did not fit after 16 attempts to grow the scratch");
            if (getenv("TFBS_DEBUG"))
                fprintf(stderr, "tfbs: block repeated (attempt %d): collided %d, need seq %llu d %llu cfg %llu vd %llu items %llu units %llu dwords %llu rows %llu rowwords %llu capr %u groups %u | caps seq %llu d %llu cfg %llu vd %llu items %llu units %llu dwords %llu rows %llu rowwords %llu capr %u groups %u\n",
                        slot->attempts, (int)collided, (unsigned long long)hp.need_seq, (unsigned long long)hp.need_d, (unsigned long long)hp.need_cfg, (unsigned long long)hp.need_vd,
                        (unsigned long long)hp.need_items, (unsigned long long)hp.need_units, (unsigned long long)hp.need_dwords, (unsigned long long)hp.need_rows,
                        (unsigned long long)hp.need_rowwords, hp.need_capr, hp.need_groups, (unsigned long long)slot->caps.seq, (unsigned long long)slot->caps.d,
                        (unsigned long long)slot->caps.cfg, (unsigned long long)slot->caps.vd, (unsigned long long)slot->caps.items, (unsigned long long)slot->caps.units,
                        (unsigned long long)slot->caps.dwords, (unsigned long long)slot->caps.rows, (unsigned long long)slot->caps.rowwords, slot->caps.capr, slot->caps.groups);
            if (collided) slot->seed = slot->seed * 0x9e3779b97f4a7c15ull + 0x7f4a7c15ull;
            int rc = quiesce(ctx);
            if (rc) return rc;
            grow_caps(hp);
            note_needs(hp);
            if ((rc = enqueue(false))) return rc;
        }
    }

    void grow_caps(const DevPlan& hp) {
        Caps& c = slot->caps;
        choose_caps(false);  // ref_items of this block
        auto g = [](uint64_t& cap, uint64_t need) { if (need > cap) cap = up(need); };
        g(c.seq, hp.need_seq);
        g(c.d, hp.need_d);
        g(c.cfg, hp.need_cfg);
        g(c.vd, hp.need_vd);
        c.items = std::max<uint64_t>(c.items, ref_items + c.vd);
        g(c.items, hp.need_items);
        g(c.units, hp.need_units);
        g(c.dwords, hp.need_dwords);
        g(c.rows, hp.need_rows);
        g(c.rowwords, hp.need_rowwords);
        g(c.terms, hp.need_terms);
        if (hp.need_capr > c.capr) c.capr = (uint32_t)up(hp.need_capr);
        if (hp.need_groups > c.groups) c.groups = groups_for(hp.need_groups);
    }
    void note_needs(const DevPlan& hp) {
        Caps& h = ctx->hint;
        h.seq = std::max<uint64_t>(h.seq, hp.need_seq);
        h.d = std::max<uint64_t>(h.d, hp.need_d);
        h.cfg = std::max<uint64_t>(h.cfg, hp.need_cfg);
        h.vd = std::max<uint64_t>(h.vd, hp.need_vd);
        h.units = std::max<uint64_t>(h.units, hp.need_units);
        h.dwords = std::max<uint64_t>(h.dwords, hp.need_dwords);
        h.rows = std::max<uint64_t>(h.rows, hp.need_rows);
        h.rowwords = std::max<uint64_t>(h.rowwords, hp.need_rowwords);
        h.terms = std::max<uint64_t>(h.terms, hp.need_terms);
        h.capr = std::max<uint32_t>(h.capr, hp.need_capr);
        h.groups = std::max<uint32_t>(h.groups, hp.need_groups);
    }

    int publish(const DevStatus& hs, const DevPlan& hp) {
        tfbs_stats& s = slot->stats;
        float t;
        if (R && S) {
            CK(cudaEventElapsedTime(&t, slot->ev_t[0], slot->ev_t[1])); s.ms_group = t;
            CK(cudaEventElapsedTime(&t, slot->ev_t[1], slot->ev_t[2])); s.ms_build = t;
            CK(cudaEventElapsedTime(&t, slot->ev_t[2], slot->ev_t[5])); s.ms_scan = t;
            CK(cudaEventElapsedTime(&t, slot->ev_t[3], slot->ev_t[4])); s.ms_scan_kernel = t;
            CK(cudaEventElapsedTime(&t, slot->ev_t[5], slot->ev_t[6])); s.ms_count = t;
        }
        CK(cudaEventElapsedTime(&t, slot->ev_t[0], slot->ev_t[6])); s.ms_total = t;
        s.n_regions = R;
        s.n_groups = hs.n_scanned;
        s.executed_cells = hs.executed_cells;
        s.nominal_cells = hs.nominal_cells;
        s.n_hits = hs.n_hits;
        s.n_keys = n_keys;
        s.n_rows = hp.n_rows;
        s.evaluated_cells = hs.evaluated_cells;
        s.n_scan_items = hp.n_items;
        s.n_dropped = hs.n_dropped;
        s.n_truncated = hs.n_truncated;
        s.reserved = (uint32_t)std::min<uint64_t>(hp.fan_keys, 0xffffffffu);
        if (getenv("TFBS_DEBUG") && hp.fan_dbg[0])
            fprintf(stderr, "tfbs: fan-out: %llu keys with a count vector, %llu pairs, %llu member updates, %llu groups / %llu samples with a non-zero difference, %llu keys in the dense pass\n",
                    (unsigned long long)hp.fan_keys, (unsigned long long)hp.fan_dbg[0], (unsigned long long)hp.fan_dbg[1], (unsigned long long)hp.fan_dbg[2],
                    (unsigned long long)hp.fan_dbg[3], (unsigned long long)hp.fan_dbg[4]);
        uint64_t table_bytes = 0;
        for (const ChunkDesc& cd : ctx->cp.chunks) table_bytes += (uint64_t)cd.tbl_words * 8 * s.scan_ctas;
        s.scan_input_bytes = (R && S) ? hp.n_units * 12 * ctx->cp.chunks.size() + table_bytes : 0;
        slot->res.n_rows = hp.n_rows;
        slot->att_cfgs = hp.n_cfg;
        slot->att_seqs = hp.n_seq;
        slot->att_terms = hp.n_terms;
        slot->res.packed_words = hp.n_rowwords;
        slot->res.row_bytes = 4;
        if (ctx->rows_width == 0) slot->res.row_bytes = hs.max_count < 256 ? 1 : (hs.max_count < 65536 ? 2 : 4);
        slot->state = 2;
        return TFBS_OK;
    }

    // row headers (both result forms)
    int fetch_headers(cudaStream_t so) {
        Results& res = slot->res;
        const uint64_t n = res.n_rows;
        CK(res.h_region.reserve(std::max<uint64_t>(1, n) * 4, false));
        CK(res.h_inner.reserve(std::max<uint64_t>(1, n) * 4, false));
        CK(res.h_pid.reserve(std::max<uint64_t>(1, n) * 2, false));
        CK(res.h_vmin.reserve(std::max<uint64_t>(1, n) * 4, false));
        CK(res.h_vmax.reserve(std::max<uint64_t>(1, n) * 4, false));
        if (n) {
            CK(cudaMemcpyAsync(res.h_region.p, slot->d_o_region.p, n * 4, cudaMemcpyDeviceToHost, so));
            CK(cudaMemcpyAsync(res.h_inner.p, slot->d_o_inner.p, n * 4, cudaMemcpyDeviceToHost, so));
            CK(cudaMemcpyAsync(res.h_pid.p, slot->d_o_pid.p, n * 2, cudaMemcpyDeviceToHost, so));
            CK(cudaMemcpyAsync(res.h_vmin.p, slot->d_o_vmin.p, n * 4, cudaMemcpyDeviceToHost, so));
            CK(cudaMemcpyAsync(res.h_vmax.p, slot->d_o_vmax.p, n * 4, cudaMemcpyDeviceToHost, so));
            slot->stats.d2h_bytes += n * 18;
        }
        return TFBS_OK;
    }

    // grouped rows -> host (stream_out: the kernels of the next block keep running meanwhile); into the caller's result arena if there is one
    int fetch_grouped() {
        Results& res = slot->res;
        if (res.have_grouped) return TFBS_OK;
        cudaStream_t so = L.stream_out;
        const uint64_t n = res.n_rows, w = res.packed_words;
        res.hg_bytes = (uint64_t)H + 1 <= 65536 ? 2 : 4;
        const bool maps = R && S;
        tfbs_arena_header* hdr = nullptr;
        slot->stats.d2h_bytes = 0;
        if (ctx->arena) {
            uint8_t* half = ctx->arena + (size_t)(slot - ctx->slot) * (ctx->arena_bytes / 2);
            hdr = reinterpret_cast<tfbs_arena_header*>(half);
            tfbs_arena_header h = *hdr;
            if (h.magic != TFBS_ARENA_MAGIC) { memset(&h, 0, sizeof h); h.magic = TFBS_ARENA_MAGIC; }
            uint64_t off = 256;
            auto place = [&](HostBuf& hb, uint64_t bytes, uint64_t* where) {
                *where = off;
                hb.bind(half + off, bytes);
                off += (bytes + 63) & ~63ull;
            };
            place(res.h_region, n * 4, &h.off_region);
            place(res.h_inner, n * 4, &h.off_inner);
            place(res.h_pid, n * 2, &h.off_pattern_id);
            place(res.h_vmin, n * 4, &h.off_vmin);
            place(res.h_vmax, n * 4, &h.off_vmax);
            place(res.h_base, n * 4, &h.off_base);
            place(res.h_bits, n, &h.off_bits);
            place(res.h_off, n * 8, &h.off_offset);
            place(res.h_packed, w * 4, &h.off_packed);
            place(res.h_ngroups, (uint64_t)(R + 1) * 8 + 8, &h.off_n_groups);
            place(res.h_hg, RH * res.hg_bytes, &h.off_hap_group);
            if (off > ctx->arena_bytes / 2)
                return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "the result arena is too small: this block needs " + std::to_string(off) + " bytes, a half of the arena has " +
                                                                std::to_string(ctx->arena_bytes / 2));
            h.n_rows = n;
            h.packed_words = w;
            h.n_samples = S;
            h.n_regions = R;
            h.hap_group_bytes = res.hg_bytes;
            h.bytes_used = off;
            const uint64_t seq = h.sequence;
            *hdr = h;
            hdr->sequence = seq;  // bumped below, once the arrays are complete
        } else {
            CK(res.h_region.reserve(std::max<uint64_t>(1, n) * 4, false));
            CK(res.h_inner.reserve(std::max<uint64_t>(1, n) * 4, false));
            CK(res.h_pid.reserve(std::max<uint64_t>(1, n) * 2, false));
            CK(res.h_vmin.reserve(std::max<uint64_t>(1, n) * 4, false));
            CK(res.h_vmax.reserve(std::max<uint64_t>(1, n) * 4, false));
            CK(res.h_base.reserve(std::max<uint64_t>(1, n) * 4, false));
            CK(res.h_bits.reserve(std::max<uint64_t>(1, n), false));
            CK(res.h_off.reserve(std::max<uint64_t>(1, n) * 8, false));
            CK(res.h_packed.reserve(std::max<uint64_t>(1, w) * 4, false));
            CK(res.h_ngroups.reserve((size_t)(R + 1) * 8 + 8, false));
            CK(res.h_hg.reserve(std::max<uint64_t>(1, RH) * res.hg_bytes, false));
        }
        if (n) {
            CK(cudaMemcpyAsync(res.h_region.p, slot->d_o_region.p, n * 4, cudaMemcpyDeviceToHost, so));
            CK(cudaMemcpyAsync(res.h_inner.p, slot->d_o_inner.p, n * 4, cudaMemcpyDeviceToHost, so));
            CK(cudaMemcpyAsync(res.h_pid.p, slot->d_o_pid.p, n * 2, cudaMemcpyDeviceToHost, so));
            CK(cudaMemcpyAsync(res.h_vmin.p, slot->d_o_vmin.p, n * 4, cudaMemcpyDeviceToHost, so));
            CK(cudaMemcpyAsync(res.h_vmax.p, slot->d_o_vmax.p, n * 4, cudaMemcpyDeviceToHost, so));
            CK(cudaMemcpyAsync(res.h_base.p, slot->d_o_base.p, n * 4, cudaMemcpyDeviceToHost, so));
            CK(cudaMemcpyAsync(res.h_bits.p, slot->d_o_bits.p, n, cudaMemcpyDeviceToHost, so));
            CK(cudaMemcpyAsync(res.h_off.p, slot->d_o_off.p, n * 8, cudaMemcpyDeviceToHost, so));
            if (w) CK(cudaMemcpyAsync(res.h_packed.p, slot->d_o_packed.p, w * 4, cudaMemcpyDeviceToHost, so));
            slot->stats.d2h_bytes += n * 31 + w * 4;
        }
        if (maps) {
            // groups per region (from the prefix array) and the haplotype -> group map, narrowed to u16 when it fits
            CK(cudaMemcpyAsync(res.h_ngroups.p, slot->d_gbase.p, (size_t)(R + 1) * 8, cudaMemcpyDeviceToHost, so));
            if (res.hg_bytes == 2) {
                int rc2 = grow(ctx, slot->d_hg_narrow, RH * 2);
                if (rc2) return rc2;
                TFBS_LAUNCH(k_narrow_groups, slot->stats.sm_count * 8, 256, 0, so)(slot->d_hap_group.as<u32>(), RH, slot->d_hg_narrow.as<u16>());
                CK(cudaMemcpyAsync(res.h_hg.p, slot->d_hg_narrow.p, RH * 2, cudaMemcpyDeviceToHost, so));
            } else {
                CK(cudaMemcpyAsync(res.h_hg.p, slot->d_hap_group.p, RH * 4, cudaMemcpyDeviceToHost, so));
            }
            slot->stats.d2h_bytes += (uint64_t)R * 4 + RH * res.hg_bytes;
        }
        CK(cudaStreamSynchronize(so));
        if (maps) {  // prefix array -> counts, in place (u64 -> u32)
            const uint64_t* gb = res.h_ngroups.as<uint64_t>();
            uint32_t* ng = res.h_ngroups.as<uint32_t>();
            for (uint32_t r = 0; r < R; ++r) ng[r] = (uint32_t)(gb[r + 1] - gb[r]);
        }
        if (hdr) {
            __atomic_thread_fence(__ATOMIC_RELEASE);
            hdr->sequence = hdr->sequence + 1;
        }
        res.have_grouped = true;
        return TFBS_OK;
    }

    // attribution -> host (stream_out), the offset arrays first: they give the sizes of the others.  Counted in d2h_bytes.  Called by the
    // collect that returns the block, while the slot's device buffers are still this block's.
    int fetch_attribution() {
        Results& res = slot->res;
        if (res.have_attribution) return TFBS_OK;
        cudaStream_t so = L.stream_out;
        const uint64_t n = res.n_rows, nc = slot->att_cfgs, ng = slot->att_seqs;
        CK(res.h_a_toff.reserve((n + 1) * 8, false));
        CK(res.h_a_croff.reserve((nc + 1) * 8, false));
        CK(res.h_a_goff.reserve((ng + 1) * 8, false));
        uint64_t* toff = res.h_a_toff.as<uint64_t>();
        uint64_t* croff = res.h_a_croff.as<uint64_t>();
        uint64_t* goff = res.h_a_goff.as<uint64_t>();
        uint64_t bytes = 0;
        auto offsets = [&](uint64_t* h, const DevBuf& d, uint64_t cnt) -> int {  // cnt = 0: the scan may not have run
            if (!cnt) { h[0] = 0; return TFBS_OK; }
            CK(cudaMemcpyAsync(h, d.p, (cnt + 1) * 8, cudaMemcpyDeviceToHost, so));
            bytes += (cnt + 1) * 8;
            return TFBS_OK;
        };
        int rc;
        if ((rc = offsets(toff, slot->d_a_toff, n)) || (rc = offsets(croff, slot->d_a_croff, nc)) || (rc = offsets(goff, slot->d_a_goff, ng))) return rc;
        CK(cudaStreamSynchronize(so));
        const uint64_t nt = toff[n], nr = croff[nc], nl = goff[ng];
        if (nt != slot->att_terms) return fail(ctx, TFBS_ERR_INTERNAL, "attribution: the term count disagrees with the gate");
        auto copy = [&](HostBuf& h, const DevBuf& d, uint64_t b) -> int {
            CK(h.reserve(std::max<uint64_t>(1, b), false));
            if (b) CK(cudaMemcpyAsync(h.p, d.p, b, cudaMemcpyDeviceToHost, so));
            bytes += b;
            return TFBS_OK;
        };
        if ((rc = copy(res.h_a_ref, slot->d_a_ref, n * 4)) || (rc = copy(res.h_a_tcfg, slot->d_a_tcfg, nt * 4)) ||
            (rc = copy(res.h_a_tdiff, slot->d_a_tdiff, nt * 4)) || (rc = copy(res.h_a_creg, slot->d_a_creg, nc * 4)) ||
            (rc = copy(res.h_a_cflags, slot->d_a_cflags, nc)) || (rc = copy(res.h_a_crec, slot->d_a_crec, nr * 4)) ||
            (rc = copy(res.h_a_gcfg, slot->d_a_gcfg, nl * 4)))
            return rc;
        CK(cudaStreamSynchronize(so));
        slot->stats.d2h_bytes += bytes;
        res.have_attribution = true;
        return TFBS_OK;
    }

    // dense rows: expanded on the device from the grouped rows, then copied
    int fetch_dense() {
        Results& res = slot->res;
        if (res.have_dense) return TFBS_OK;
        cudaStream_t so = L.stream_out;
        const uint64_t n = res.n_rows;
        const uint32_t eb = res.row_bytes;
        int rc;
        slot->stats.d2h_bytes = 0;
        if ((rc = fetch_headers(so))) return rc;
        CK(res.h_left.reserve(std::max<uint64_t>(1, n * S) * eb, false));
        CK(res.h_right.reserve(std::max<uint64_t>(1, n * S) * eb, false));
        if (n && S) {
            if ((rc = grow(ctx, slot->d_left, n * S * eb))) return rc;
            if ((rc = grow(ctx, slot->d_right, n * S * eb))) return rc;
            DevDenseRows out{slot->d_left.p, slot->d_right.p};
            const u64* n_rows_ptr = &slot->d_plan.as<DevPlan>()->n_rows;
#define TFBS_EXPAND(T)                                                                                                                     \
    TFBS_LAUNCH(k_rows_expand<T>, grid_for(n * 32, 256), 256, 0, so)(S, H, slot->d_hap_group.as<u32>(), n_rows_ptr, slot->d_o_region.as<u32>(), \
                                                                      slot->d_o_base.as<u32>(), slot->d_o_bits.as<u8>(), slot->d_o_off.as<u64>(),  \
                                                                      slot->d_o_packed.as<u32>(), out)
            if (eb == 1) TFBS_EXPAND(u8);
            else if (eb == 2) TFBS_EXPAND(u16);
            else TFBS_EXPAND(u32);
#undef TFBS_EXPAND
            CK(cudaMemcpyAsync(res.h_left.p, slot->d_left.p, n * S * eb, cudaMemcpyDeviceToHost, so));
            CK(cudaMemcpyAsync(res.h_right.p, slot->d_right.p, n * S * eb, cudaMemcpyDeviceToHost, so));
            slot->stats.d2h_bytes += 2 * n * S * eb;
        }
        CK(cudaStreamSynchronize(so));
        res.have_dense = true;
        return TFBS_OK;
    }
};

}  // namespace
