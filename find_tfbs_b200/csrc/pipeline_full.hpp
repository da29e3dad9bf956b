// pipeline_full.hpp -- the full scan: every distinct haplotype of every region scored in full, like the reference (main.rs:101-147)
// Host side of libtfbs_b200.so (tfbs.cu is the map); one translation unit.
//
// Used when option "delta" = 0, when the hit list is recorded ("record_matches", tfbs_get_matches) and by tfbs_audit_block.  It runs
// a block to completion (sizes come back to the host between the phases, regions go through the scratch in batches) and keeps one
// dense count row per distinct haplotype: the shape of the reference's own algorithm, and the yardstick of the scan kernel's roofline.
// The default path is pipeline_config.hpp.
#pragma once
#include "host_common.hpp"

namespace {

struct FullPipeline {
    tfbs_ctx* ctx;
    Slot* slot;
    Lane& L;  // lane 0: the full scan owns the device
    BlockDev& B;
    Results& res;
    cudaStream_t st;
    const uint32_t R, S, H;
    const uint64_t RH;
    DevStatus* dst = nullptr;
    DevBlock db{};
    DevMatches dm{};
    DevConfigs no_cf{};
    uint32_t n_pid = 0;
    int smem_bytes = 0;
    bool wide = false;
    uint32_t scan_grid = 0;
    // accumulated over the batches
    float ms_build = 0, ms_scan = 0, ms_count = 0, ms_scan_kernel = 0;
    uint64_t n_items_total = 0;

    // a batch of regions [r0, r1) and the sizes its scratch arrays are planned for
    struct Batch {
        uint32_t r0 = 0, r1 = 0, nr = 0;
        uint64_t n_seq = 0, n_d = 0, n_units = 0, n_c = 0, n_keys = 0;
        DevSeqs sq{};
        DevRefHits drh{};
        DevCounts dc{};
        const u64* d_n_items = nullptr;
        uint64_t n_list_host = 0;
        DevStatus hs{};  // status word after the batch's rows pass
    };

    FullPipeline(tfbs_ctx* c, Slot* s)
        : ctx(c), slot(s), L(c->lane[s->lane]), B(*s->in), res(s->res), st(L.stream), R(s->in->R), S(s->in->S), H(s->in->H), RH((uint64_t)s->in->R * s->in->H) {}

    int run() {
        int rc;
        if ((rc = begin())) return rc;
        if (R == 0 || S == 0) {
            CK(cudaStreamSynchronize(st));
            return TFBS_OK;
        }
        if ((rc = encode_inputs())) return rc;
        if ((rc = group_haplotypes())) return rc;
        if ((rc = region_prefixes())) return rc;
        if ((rc = setup_scan())) return rc;
        for (uint32_t r0 = 0; r0 < R;) {
            Batch b;
            if ((rc = plan_batch(r0, &b))) return rc;
            if ((rc = reserve_batch(&b))) return rc;
            CK(cudaEventRecord(ctx->ev[2], st));
            if ((rc = build_sequences(b))) return rc;
            CK(cudaEventRecord(ctx->ev[3], st));
            if ((rc = scan_pass(&b))) return rc;
            CK(cudaEventRecord(ctx->ev[4], st));
            if ((rc = count_and_filter(&b))) return rc;
            if ((rc = fetch_rows(b))) return rc;
            if ((rc = batch_timers())) return rc;
            r0 = b.r1;
        }
        return finish();
    }

private:
    tfbs_stats& stats() { return slot->stats; }
    uint32_t& launches() { return slot->stats.total_launches; }

    int scan(const uint32_t* d_in, uint64_t n, u64* d_out) { return device_scan(ctx, L, d_in, n, nullptr, d_out, &launches()); }

    int read_status(DevStatus* hs) {
        CK(cudaMemcpyAsync(slot->h_status.p, dst, sizeof(DevStatus), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        memcpy(hs, slot->h_status.p, sizeof *hs);
        return TFBS_OK;
    }

    int begin() {
        memset(&slot->stats, 0, sizeof slot->stats);
        stats().h2d_bytes = B.h2d_bytes;
        stats().sm_count = (uint32_t)ctx->prop.multiProcessorCount;
        res.n_rows = 0;
        res.have_dense = true;
        res.have_grouped = false;
        res.row_bytes = 4;
        ctx->n_matches = 0;
        ctx->matches_truncated = false;
        int rc;
        if ((rc = quiesce(ctx))) return rc;  // this pipeline owns the device for the duration of the call
        if ((rc = reserve_encoding(ctx, L, B))) return rc;
        CK(slot->d_status.reserve(sizeof(DevStatus)));
        CK(slot->h_status.reserve(sizeof(DevStatus), false));
        CK(ctx->h_totals.reserve(64, false));
        dst = slot->d_status.as<DevStatus>();
        DevStatus init{};
        init.err_key = ~0ull;
        init.bad_ref_base = ~0ull;
        init.bad_allele_base = ~0ull;
        memcpy(slot->h_status.p, &init, sizeof init);
        CK(cudaMemcpyAsync(dst, slot->h_status.p, sizeof init, cudaMemcpyHostToDevice, st));
        CK(cudaEventRecord(ctx->ev[0], st));
        return TFBS_OK;
    }

    // ASCII -> nucleotide codes, Diff classes, prefix hashes of the reference windows
    int encode_inputs() {
        if (B.n_ref_bytes) {
            TFBS_LAUNCH(k_encode, std::min<unsigned>(grid_for(B.n_ref_bytes, 256), stats().sm_count * 16), 256, 0, st)(B.d_ref_ascii.as<u8>(), L.d_ref_codes.as<u8>(),
                                                                                                     B.n_ref_bytes, &dst->bad_ref_base);
            ++launches();
        }
        if (B.n_allele_bytes) {
            TFBS_LAUNCH(k_encode, std::min<unsigned>(grid_for(B.n_allele_bytes, 256), stats().sm_count * 16), 256, 0, st)(
                B.d_allele_ascii.as<u8>(), L.d_allele_codes.as<u8>(), B.n_allele_bytes, &dst->bad_allele_base);
            ++launches();
        }
        db = dev_block(L, B);
        TFBS_LAUNCH(k_variant_prep, R, 128, 0, st)(db, 0, L.d_var_class.as<u32>(), L.d_var_inwin.as<u8>(), (u32*)nullptr);
        TFBS_LAUNCH(k_ref_prefix, R, SCAN_THREADS, 0, st)(db, 0, L.d_ref_prefix.as<u64>());
        launches() += 2;
        return TFBS_OK;
    }

    // ---- phase 1: grouping (K0), over super-batches bounded by the hash table; a signature collision retries with another seed ----
    int group_haplotypes() {
        CK(L.d_sig.reserve(RH * 8));
        CK(L.d_nd_in.reserve(RH * 4));
        CK(L.d_leader.reserve(RH * 4));
        CK(L.d_hap_group.reserve(RH * 4));
        CK(L.d_ngroups.reserve((size_t)R * 4));
        CK(L.d_sum_nd.reserve((size_t)R * 4));
        CK(L.d_ref_used.reserve((size_t)R * 4));
        if (ctx->audit) CK(L.d_hap_flags.reserve(RH));
        const uint64_t max_pairs = 1ull << 25;
        uint32_t regions_per_super = (uint32_t)std::max<uint64_t>(1, max_pairs / std::max<uint32_t>(1, H));
        uint64_t seed = 0x243f6a8885a308d3ull;
        for (int attempt = 0;; ++attempt) {
            for (uint32_t r0 = 0; r0 < R; r0 += regions_per_super) {
                uint32_t nr = std::min(regions_per_super, R - r0);
                uint64_t pairs = (uint64_t)nr * H;
                uint32_t cap = 1024;
                while (cap < 2 * pairs) cap <<= 1;
                CK(L.d_keys.reserve((size_t)cap * 8));
                CK(L.d_vals.reserve((size_t)cap * 4));
                CK(cudaMemsetAsync(L.d_keys.p, 0, (size_t)cap * 8, st));
                CK(cudaMemsetAsync(L.d_vals.p, 0xff, (size_t)cap * 4, st));
                TFBS_LAUNCH(k_signatures, grid_for((uint64_t)nr * ((H + 31) / 32) * 32, 256), 256, 0, st)(db, r0, nr, seed, L.d_sig.as<u64>(), L.d_nd_in.as<u32>());
                TFBS_LAUNCH(k_group_insert, grid_for(pairs, 256), 256, 0, st)(H, r0, nr, L.d_sig.as<u64>(), L.d_keys.as<u64>(), L.d_vals.as<u32>(), cap - 1, 0u);
                TFBS_LAUNCH(k_group_lookup, grid_for(pairs, 256), 256, 0, st)(db, r0, nr, L.d_sig.as<u64>(), L.d_keys.as<u64>(), L.d_vals.as<u32>(), cap - 1, 0u,
                                                                     L.d_leader.as<u32>(), dst);
                TFBS_LAUNCH(k_group_rank, nr, 256, 0, st)(H, r0, L.d_leader.as<u32>(), L.d_nd_in.as<u32>(), L.d_hap_group.as<u32>(),
                                                 L.d_ngroups.as<u32>(), L.d_sum_nd.as<u32>());
                launches() += 4;
            }
            CK(cudaGetLastError());
            ctx->h_ngroups.resize(R);
            ctx->h_sum_nd.resize(R);
            CK(cudaMemcpyAsync(ctx->h_ngroups.data(), L.d_ngroups.p, (size_t)R * 4, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(ctx->h_sum_nd.data(), L.d_sum_nd.p, (size_t)R * 4, cudaMemcpyDeviceToHost, st));
            DevStatus hs;
            int rc = read_status(&hs);
            if (rc) return rc;
            if (hs.bad_ref_base != ~0ull || hs.bad_allele_base != ~0ull) {
                // util.rs:15 panic!("Unknown nucleotide {}", l)
                return fail(ctx, TFBS_ERR_UNKNOWN_NUCLEOTIDE,
                            std::string("Unknown nucleotide at byte ") +
                                std::to_string(hs.bad_ref_base != ~0ull ? hs.bad_ref_base : hs.bad_allele_base) +
                                (hs.bad_ref_base != ~0ull ? " of ref_bases" : " of allele_bases"));
            }
            if (hs.sig_collision == 0 || !ctx->verify_groups) break;
            if (attempt >= 3) return fail(ctx, TFBS_ERR_INTERNAL, "haplotype signature hash collision persisted over 4 seeds");
            seed = seed * 0x9e3779b97f4a7c15ull + 0x7f4a7c15ull;
            CK(cudaMemsetAsync(&dst->sig_collision, 0, 4, st));
        }
        CK(cudaEventRecord(ctx->ev[1], st));
        return TFBS_OK;
    }

    // per region: first sequence (gbase), first count word (cbase) and first key (kbase), block-wide
    int region_prefixes() {
        n_pid = (uint32_t)ctx->cp.pid_list.size();
        ctx->h_gbase.assign(R + 1, 0);
        ctx->h_cbase.assign(R + 1, 0);
        ctx->h_kbase.assign(R + 1, 0);
        for (uint32_t r = 0; r < R; ++r) {
            uint64_t nk = B.h_inner_off[r + 1] - B.h_inner_off[r];
            ctx->h_gbase[r + 1] = ctx->h_gbase[r] + ctx->h_ngroups[r];
            ctx->h_cbase[r + 1] = ctx->h_cbase[r] + (uint64_t)ctx->h_ngroups[r] * n_pid * nk;
            ctx->h_kbase[r + 1] = ctx->h_kbase[r] + (uint64_t)n_pid * nk;
        }
        int rc;
        if ((rc = upload_on(ctx, st, L.d_gbase, ctx->h_gbase.data(), R + 1, nullptr))) return rc;
        if ((rc = upload_on(ctx, st, L.d_cbase, ctx->h_cbase.data(), R + 1, nullptr))) return rc;
        if ((rc = upload_on(ctx, st, L.d_kbase, ctx->h_kbase.data(), R + 1, nullptr))) return rc;
        return TFBS_OK;
    }

    // match buffer, shared-memory size and grid of the scan kernel
    int setup_scan() {
        if (ctx->record_matches) {
            CK(L.d_m_region.reserve(ctx->max_matches * 4));
            CK(L.d_m_pattern.reserve(ctx->max_matches * 4));
            CK(L.d_m_group.reserve(ctx->max_matches * 4));
            CK(L.d_m_start.reserve(ctx->max_matches * 8));
        }
        dm.enabled = ctx->record_matches ? 1u : 0u;
        dm.cap = (u32)std::min<uint64_t>(ctx->max_matches, 0xffffffffu);
        dm.region = L.d_m_region.as<u32>();
        dm.pattern_index = L.d_m_pattern.as<u32>();
        dm.group = L.d_m_group.as<u32>();
        dm.start = L.d_m_start.as<i64>();
        smem_bytes = (int)(sizeof(CtaShared) + SCAN_WARPS * sizeof(WarpShared) + ((ctx->cp.max_chunk_bytes + 15) & ~15u));
        wide = ctx->cp.fields == 2;
        if (wide) CK(raise_smem_limit(k_scan<2>, ctx->device, smem_bytes));
        else CK(raise_smem_limit(k_scan<3>, ctx->device, smem_bytes));
        scan_grid = (uint32_t)ctx->prop.multiProcessorCount;  // persistent: one CTA per SM shares one copy of the tables
        if (ctx->scan_ctas_per_sm < 0) scan_grid = (uint32_t)std::max(1, -ctx->scan_ctas_per_sm);  // debugging: fixed grid size
        stats().scan_ctas = scan_grid;
        return TFBS_OK;
    }

    // ---- phase 2: batches under the scratch budget ---------------------------------------------------
    void region_cost(uint32_t r, uint64_t* n_seq, uint64_t* n_d, uint64_t* n_units, uint64_t* n_c, uint64_t* n_keys) const {
        uint64_t g = ctx->h_ngroups[r];
        uint64_t W = (uint64_t)(B.h_region_end[r] - B.h_region_start[r] + 1) + B.h_ins_extra[r];
        uint64_t nk = B.h_inner_off[r + 1] - B.h_inner_off[r];
        *n_seq = g;
        *n_d = ctx->h_sum_nd[r];
        *n_units = g * ((W + 31) / 32 + 3);
        *n_c = g * n_pid * nk;
        *n_keys = (uint64_t)n_pid * nk;
    }
    static uint64_t bytes_of(uint64_t n_seq, uint64_t n_d, uint64_t n_units, uint64_t n_c, uint64_t n_keys) {
        // sequences (with one work-list item each), diff lists + segments, packed bases, counts, keys, the sequence-keyed map
        return n_seq * (4 * 7 + 8 * 3 + 1 + 32 + 40) + n_d * (4 + 32) + n_units * 12 + n_c * 4 + n_keys * 24 + n_seq * 2 * 12;
    }

    int plan_batch(uint32_t r0, Batch* b) {
        b->r0 = r0;
        uint32_t r1 = r0;
        while (r1 < R) {
            uint64_t a, b2, c2, d2, e2;
            region_cost(r1, &a, &b2, &c2, &d2, &e2);
            if (r1 > r0 && (bytes_of(b->n_seq + a, b->n_d + b2, b->n_units + c2, b->n_c + d2, b->n_keys + e2) > ctx->scratch_bytes ||
                            b->n_seq + a > 0x7fffffffull || b->n_seq + a + b->n_d + b2 > (1ull << 30)))
                break;
            b->n_seq += a; b->n_d += b2; b->n_units += c2; b->n_c += d2; b->n_keys += e2;
            ++r1;
        }
        b->r1 = r1;
        b->nr = r1 - r0;
        if (b->n_seq > 0x7fffffffull || b->n_seq + b->n_d > (1ull << 30))
            return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "a single region has more haplotype groups / carried variants than one batch can hold");
        return TFBS_OK;
    }

    int reserve_batch(Batch* b) {
        const uint64_t n_seq = b->n_seq, n_d = b->n_d, n_c = b->n_c, n_keys = b->n_keys;
        const uint64_t ic = std::max<uint64_t>(1, n_seq);  // at most one item per sequence
        CK(L.d_seq_region.reserve(n_seq * 4));
        CK(L.d_seq_leader.reserve(n_seq * 4));
        CK(L.d_seq_nd.reserve(n_seq * 4));
        CK(L.d_seq_doff.reserve((n_seq + 1) * 8));
        CK(L.d_dlist.reserve(std::max<uint64_t>(1, n_d) * 4));
        CK(L.d_segs.reserve((2 * n_d + 2 * n_seq) * sizeof(Seg)));
        CK(L.d_seq_nseg.reserve(n_seq * 4));
        CK(L.d_seq_len.reserve(n_seq * 4));
        CK(L.d_seq_hash.reserve(n_seq * 8));
        CK(L.d_seq_flags.reserve(n_seq));
        CK(L.d_seq_ntake.reserve(n_seq * 4));
        CK(L.d_C.reserve(std::max<uint64_t>(1, n_c) * 4));
        CK(L.d_vmin.reserve(std::max<uint64_t>(1, n_keys) * 4));
        CK(L.d_vmax.reserve(std::max<uint64_t>(1, n_keys) * 4));
        CK(L.d_flag.reserve(std::max<uint64_t>(1, n_keys) * 4));
        CK(L.d_rowidx.reserve((n_keys + 1) * 8));
        CK(L.d_refcnt.reserve((size_t)b->nr * 4));
        CK(L.d_seq_nitems.reserve(n_seq * 4));
        CK(L.d_item_off.reserve((n_seq + 1) * 8));
        CK(L.d_items.reserve(ic * sizeof(ScanItem)));
        CK(L.d_list.reserve(ic * 4));
        CK(L.d_ent_units.reserve(ic * 4));
        CK(L.d_ent_uoff.reserve((ic + 1) * 8));
        CK(L.d_pk.reserve(std::max<uint64_t>(1, b->n_units) * 8));
        CK(L.d_nm.reserve(std::max<uint64_t>(1, b->n_units) * 4));

        DevSeqs& sq = b->sq;
        sq = DevSeqs{};
        sq.n_seq = (u32)n_seq;
        sq.gbase = L.d_gbase.as<u64>();
        sq.gbase0 = ctx->h_gbase[b->r0];
        sq.seq_region = L.d_seq_region.as<u32>();
        sq.seq_leader = L.d_seq_leader.as<u32>();
        sq.seq_nd = L.d_seq_nd.as<u32>();
        sq.seq_doff = L.d_seq_doff.as<u64>();
        sq.dlist = L.d_dlist.as<u32>();
        sq.segs = L.d_segs.as<Seg>();
        sq.seq_nseg = L.d_seq_nseg.as<u32>();
        sq.seq_len = L.d_seq_len.as<u32>();
        sq.ent_units = L.d_ent_units.as<u32>();
        sq.ent_uoff = L.d_ent_uoff.as<u64>();
        sq.pk = L.d_pk.as<u64>();
        sq.nm = L.d_nm.as<u32>();
        sq.seq_hash = L.d_seq_hash.as<u64>();
        sq.seq_flags = L.d_seq_flags.as<u8>();
        sq.seq_ntake = L.d_seq_ntake.as<u32>();
        sq.seq_nitems = L.d_seq_nitems.as<u32>();
        sq.item_off = L.d_item_off.as<u64>();
        sq.items = L.d_items.as<ScanItem>();
        sq.n_items_cap = (u32)std::min<uint64_t>(ic, 0xffffffffu);
        sq.units_cap = b->n_units;
        b->drh = DevRefHits{nullptr, L.d_refcnt.as<u32>(), 0, b->r0};
        b->dc.C = L.d_C.as<u32>();
        b->dc.cbase = L.d_cbase.as<u64>();
        b->dc.cbase0 = ctx->h_cbase[b->r0];
        b->d_n_items = sq.item_off + n_seq;
        return TFBS_OK;
    }

    // K1: segments + hash of every distinct haplotype, then the sequence-keyed map of load_haplotypes
    int build_sequences(Batch& b) {
        int rc;
        const uint64_t n_seq = b.n_seq;
        TFBS_LAUNCH(k_seq_init, b.nr, 128, 0, st)(H, b.r0, L.d_hap_group.as<u32>(), L.d_leader.as<u32>(), L.d_nd_in.as<u32>(), b.sq);
        ++launches();
        if ((rc = scan(b.sq.seq_nd, n_seq, b.sq.seq_doff))) return rc;
        TFBS_LAUNCH(k_walk, grid_for(n_seq, 128), 128, 0, st)(db, b.sq, ~0ull, dst, 1u);
        ++launches();
        uint32_t cap = 1024;
        while (cap < 2 * n_seq) cap <<= 1;
        CK(L.d_keys.reserve((size_t)cap * 8));
        CK(L.d_vals.reserve((size_t)cap * 4));
        CK(cudaMemsetAsync(L.d_keys.p, 0, (size_t)cap * 8, st));
        CK(cudaMemsetAsync(L.d_vals.p, 0xff, (size_t)cap * 4, st));
        CK(cudaMemsetAsync(L.d_ref_used.as<u32>() + b.r0, 0, (size_t)b.nr * 4, st));
        TFBS_LAUNCH(k_seq_insert, grid_for(n_seq, 256), 256, 0, st)(b.sq, L.d_keys.as<u64>(), L.d_vals.as<u32>(), cap - 1, 0u, 0u);
        TFBS_LAUNCH(k_seq_resolve, grid_for(n_seq, 128), 128, 0, st)(db, b.sq, L.d_keys.as<u64>(), L.d_vals.as<u32>(), cap - 1, 0u, 0u, dst, 1u);
        TFBS_LAUNCH(k_redirect, grid_for((uint64_t)b.nr * H, 256), 256, 0, st)(H, b.r0, b.nr, b.sq, L.d_hap_group.as<u32>(), L.d_ref_used.as<u32>(),
                                                                        ctx->audit ? L.d_hap_flags.as<u8>() : nullptr, (u64*)nullptr, 0u, 0u, 0ull, 0u, (const u32*)nullptr);
        launches() += 3;
        return TFBS_OK;
    }

    // K2: one item per scanned sequence, packing of its bases, the scan (one launch per pattern chunk)
    int scan_pass(Batch* bp) {
        Batch& b = *bp;
        DevSeqs& sq = b.sq;
        int rc;
        const uint64_t n_seq = b.n_seq;
        if (b.n_c) CK(cudaMemsetAsync(L.d_C.p, 0, b.n_c * 4, st));
        TFBS_LAUNCH(k_full_items<false>, grid_for(n_seq, 128), 128, 0, st)(sq, L.d_ref_used.as<u32>());
        ++launches();
        if ((rc = scan(sq.seq_nitems, n_seq, sq.item_off))) return rc;
        TFBS_LAUNCH(k_full_items<true>, grid_for(n_seq, 128), 128, 0, st)(sq, L.d_ref_used.as<u32>());
        TFBS_LAUNCH(k_vitem_units, grid_for(n_seq, 256), 256, 0, st)(sq, b.d_n_items, L.d_list.as<u32>());
        launches() += 2;
        if ((rc = device_scan(ctx, L, sq.ent_units, n_seq, b.d_n_items, sq.ent_uoff, &launches()))) return rc;
        CK(cudaMemcpyAsync((char*)ctx->h_totals.p + 24, b.d_n_items, 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        b.n_list_host = ctx->h_totals.as<uint64_t>()[3];
        uint64_t table_bytes = 0;
        if (b.n_list_host) {
            TFBS_LAUNCH(k_emit_list, grid_for(b.n_list_host * EMIT_LANES, 256), 256, 0, st)(db, sq, L.d_list.as<u32>(), b.d_n_items);
            TFBS_LAUNCH(k_item_stats, grid_for(b.n_list_host, 256), 256, 0, st)(sq, ctx->dpat, L.d_list.as<u32>(), b.d_n_items, dst);
            launches() += 2;
        }
        CK(cudaEventRecord(ctx->ev[8], st));
        for (uint32_t c = 0; c < ctx->cp.chunks.size() && b.n_list_host; ++c) {
            CK(cudaMemsetAsync(&dst->work_counter, 0, 4, st));
            if (wide) TFBS_LAUNCH(k_scan<2>, scan_grid, SCAN_CTA, smem_bytes, st)(db, sq, ctx->dpat, b.dc, dm, b.drh, no_cf, 0, L.d_list.as<u32>(), b.d_n_items, 1u, dst, c);
            else TFBS_LAUNCH(k_scan<3>, scan_grid, SCAN_CTA, smem_bytes, st)(db, sq, ctx->dpat, b.dc, dm, b.drh, no_cf, 0, L.d_list.as<u32>(), b.d_n_items, 1u, dst, c);
            ++launches();
            ++stats().scan_launches;
            table_bytes += (uint64_t)ctx->cp.chunks[c].tbl_words * 8 * scan_grid;
        }
        CK(cudaEventRecord(ctx->ev[9], st));
        CK(cudaGetLastError());
        // algorithmic input of the scan launches: 12 B per unit of 32 packed bases, once per pattern chunk, plus the tables once per CTA
        CK(cudaMemcpyAsync((char*)ctx->h_totals.p + 32, sq.ent_uoff + std::min<uint64_t>(b.n_list_host, n_seq), 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        stats().scan_input_bytes += ctx->h_totals.as<uint64_t>()[4] * 12 * ctx->cp.chunks.size() + table_bytes;
        return TFBS_OK;
    }

    // min / max per key and the row index of every emitted key; the row count lands in h_totals[0]
    int rows_pass(Batch& b) {
        if (!b.n_keys) return TFBS_OK;
        int rc;
        TFBS_LAUNCH(k_rows_minmax, b.nr, 128, 0, st)(db, b.r0, L.d_hap_group.as<u32>(), b.dc, L.d_gbase.as<u64>(), n_pid, L.d_kbase.as<u64>(),
                                          ctx->h_kbase[b.r0], ctx->rows_mode, L.d_vmin.as<u32>(), L.d_vmax.as<u32>(), L.d_flag.as<u32>(),
                                          &dst->max_count);
        ++launches();
        if ((rc = scan(L.d_flag.as<u32>(), b.n_keys, L.d_rowidx.as<u64>()))) return rc;
        CK(cudaMemcpyAsync(ctx->h_totals.p, L.d_rowidx.as<u64>() + b.n_keys, 8, cudaMemcpyDeviceToHost, st));
        return TFBS_OK;
    }

    // K3 up to the row count; reports the reference's panics
    int count_and_filter(Batch* bp) {
        Batch& b = *bp;
        int rc;
        TFBS_LAUNCH(k_nominal, grid_for((uint64_t)b.nr * H, 256), 256, 0, st)(db, b.r0, b.nr, L.d_hap_group.as<u32>(), b.sq, ctx->dpat, dst);
        TFBS_LAUNCH(k_seq_stats, grid_for(b.n_seq, 256), 256, 0, st)(b.sq, ctx->dpat, L.d_ref_used.as<u32>(), dst);
        launches() += 2;
        if ((rc = rows_pass(b))) return rc;
        if ((rc = read_status(&b.hs))) return rc;
        CK(cudaGetLastError());
        const DevStatus& hs = b.hs;
        if (hs.err_key != ~0ull) {
            uint32_t q = (uint32_t)(hs.err_key >> 32);
            // region of sequence q: last r with gbase[r] - gbase[r0] <= q
            uint32_t r = (uint32_t)(std::upper_bound(ctx->h_gbase.begin() + b.r0, ctx->h_gbase.begin() + b.r1, ctx->h_gbase[b.r0] + q) - ctx->h_gbase.begin() - 1);
            return patch_panic(ctx, hs.err_key, r, B.h_region_start[r]);
        }
        if (hs.seq_collision) return fail(ctx, TFBS_ERR_INTERNAL, "sequence hash collision between distinct haplotypes");
        n_items_total += b.n_list_host;
        return TFBS_OK;
    }

    // compaction of the emitted rows and their copy into the pinned result buffers (appended to the rows of earlier batches)
    int fetch_rows(Batch& b) {
        const uint64_t batch_rows = b.n_keys ? *ctx->h_totals.as<uint64_t>() : 0;
        if (batch_rows) {
            const uint64_t n_keys = b.n_keys;
            uint64_t tot = res.n_rows + batch_rows;
            // element width of left / right: u32 like the reference's Vec<u32>, or (option rows_width = 0) the narrowest type that
            // holds every count of the block: the rows are the dominant PCIe traffic of large cohorts
            uint32_t eb = 4;
            if (ctx->rows_width == 0) eb = b.hs.max_count < 256 ? 1 : (b.hs.max_count < 65536 ? 2 : 4);
            if (res.n_rows == 0) res.row_bytes = eb;
            if (eb > res.row_bytes) {  // an earlier batch of this block was stored narrower: widen it in place (rare)
                const uint64_t n = res.n_rows * S;
                CK(res.h_left.reserve(tot * S * eb, true));
                CK(res.h_right.reserve(tot * S * eb, true));
                for (HostBuf* hb : {&res.h_left, &res.h_right})
                    for (uint64_t i = n; i-- > 0;) {
                        uint32_t v = res.row_bytes == 1 ? hb->as<uint8_t>()[i] : hb->as<uint16_t>()[i];
                        if (eb == 2) hb->as<uint16_t>()[i] = (uint16_t)v; else hb->as<uint32_t>()[i] = v;
                    }
                res.row_bytes = eb;
            }
            eb = res.row_bytes;
            CK(L.d_rows_region.reserve(batch_rows * 4));
            CK(L.d_rows_inner.reserve(batch_rows * 4));
            CK(L.d_rows_pid.reserve(batch_rows * 2));
            CK(L.d_rows_vmin.reserve(batch_rows * 4));
            CK(L.d_rows_vmax.reserve(batch_rows * 4));
            CK(L.d_rows_left.reserve(batch_rows * S * eb));
            CK(L.d_rows_right.reserve(batch_rows * S * eb));
            CK(res.h_region.reserve(tot * 4, true));
            CK(res.h_inner.reserve(tot * 4, true));
            CK(res.h_pid.reserve(tot * 2, true));
            CK(res.h_vmin.reserve(tot * 4, true));
            CK(res.h_vmax.reserve(tot * 4, true));
            CK(res.h_left.reserve(tot * S * eb, true));
            CK(res.h_right.reserve(tot * S * eb, true));
            DevRows dr{L.d_rows_region.as<u32>(), L.d_rows_inner.as<u32>(), L.d_rows_pid.as<u16>(), L.d_rows_vmin.as<u32>(),
                       L.d_rows_vmax.as<u32>(), L.d_rows_left.p, L.d_rows_right.p};
#define TFBS_ROWS_WRITE(T)                                                                                                              \
    TFBS_LAUNCH(k_rows_write<T>, grid_for(n_keys * 32, 256), 256, 0, st)(db, b.r0, b.nr, L.d_hap_group.as<u32>(), b.dc, n_pid, ctx->d_pid_list.as<u16>(), \
                                                                L.d_kbase.as<u64>(), ctx->h_kbase[b.r0], n_keys, L.d_vmin.as<u32>(),   \
                                                                L.d_vmax.as<u32>(), L.d_flag.as<u32>(), L.d_rowidx.as<u64>(), dr, 0)
            if (eb == 1) TFBS_ROWS_WRITE(u8);
            else if (eb == 2) TFBS_ROWS_WRITE(u16);
            else TFBS_ROWS_WRITE(u32);
#undef TFBS_ROWS_WRITE
            ++launches();
            uint64_t o = res.n_rows;
            CK(cudaMemcpyAsync(res.h_region.as<u32>() + o, dr.region, batch_rows * 4, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(res.h_inner.as<u32>() + o, dr.inner, batch_rows * 4, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(res.h_pid.as<u16>() + o, dr.pattern_id, batch_rows * 2, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(res.h_vmin.as<u32>() + o, dr.vmin, batch_rows * 4, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(res.h_vmax.as<u32>() + o, dr.vmax, batch_rows * 4, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(res.h_left.as<uint8_t>() + o * S * eb, dr.left, batch_rows * S * eb, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(res.h_right.as<uint8_t>() + o * S * eb, dr.right, batch_rows * S * eb, cudaMemcpyDeviceToHost, st));
            stats().d2h_bytes += batch_rows * (4 * 4 + 2 + 2ull * eb * S);
            res.n_rows = tot;
        }
        CK(cudaEventRecord(ctx->ev[5], st));
        CK(cudaStreamSynchronize(st));
        return TFBS_OK;
    }

    int batch_timers() {
        float t;
        CK(cudaEventElapsedTime(&t, ctx->ev[2], ctx->ev[3]));
        ms_build += t;
        CK(cudaEventElapsedTime(&t, ctx->ev[3], ctx->ev[4]));
        ms_scan += t;
        CK(cudaEventElapsedTime(&t, ctx->ev[4], ctx->ev[5]));
        ms_count += t;
        CK(cudaEventElapsedTime(&t, ctx->ev[8], ctx->ev[9]));
        ms_scan_kernel += t;
        return TFBS_OK;
    }

    // final status word, the match list and the audit flags, timings and counters of the run
    int finish() {
        CK(cudaEventRecord(ctx->ev[6], st));
        if (ctx->record_matches) {
            CK(ctx->h_hap_group.reserve(RH * 4, false));
            CK(cudaMemcpyAsync(ctx->h_hap_group.p, L.d_hap_group.p, RH * 4, cudaMemcpyDeviceToHost, st));
        }
        if (ctx->audit) {
            CK(ctx->h_hap_flags.reserve(RH, false));
            CK(cudaMemcpyAsync(ctx->h_hap_flags.p, L.d_hap_flags.p, RH, cudaMemcpyDeviceToHost, st));
        }
        DevStatus hs;
        int rc = read_status(&hs);
        if (rc) return rc;
        if (ctx->record_matches) {
            uint64_t n = std::min<uint64_t>(hs.n_matches, dm.cap);
            ctx->matches_truncated = hs.n_matches > dm.cap;
            ctx->n_matches_found = hs.n_matches;
            CK(ctx->h_m_region.reserve(std::max<uint64_t>(1, n) * 4, false));
            CK(ctx->h_m_pattern.reserve(std::max<uint64_t>(1, n) * 4, false));
            CK(ctx->h_m_group.reserve(std::max<uint64_t>(1, n) * 4, false));
            CK(ctx->h_m_start.reserve(std::max<uint64_t>(1, n) * 8, false));
            if (n) {
                CK(cudaMemcpyAsync(ctx->h_m_region.p, dm.region, n * 4, cudaMemcpyDeviceToHost, st));
                CK(cudaMemcpyAsync(ctx->h_m_pattern.p, dm.pattern_index, n * 4, cudaMemcpyDeviceToHost, st));
                CK(cudaMemcpyAsync(ctx->h_m_group.p, dm.group, n * 4, cudaMemcpyDeviceToHost, st));
                CK(cudaMemcpyAsync(ctx->h_m_start.p, dm.start, n * 8, cudaMemcpyDeviceToHost, st));
                CK(cudaStreamSynchronize(st));
            }
            ctx->n_matches = n;
        }
        float t;
        CK(cudaEventElapsedTime(&t, ctx->ev[0], ctx->ev[1]));
        stats().ms_group = t;
        CK(cudaEventElapsedTime(&t, ctx->ev[0], ctx->ev[6]));
        stats().ms_total = t;
        stats().ms_build = ms_build;
        stats().ms_scan = ms_scan;
        stats().ms_count = ms_count;
        stats().n_regions = R;
        stats().n_groups = hs.n_scanned;
        stats().executed_cells = hs.executed_cells;
        stats().nominal_cells = hs.nominal_cells;
        stats().n_hits = hs.n_hits;
        stats().n_keys = ctx->h_kbase[R];
        stats().n_rows = res.n_rows;
        stats().evaluated_cells = hs.evaluated_cells;
        stats().n_scan_items = n_items_total;
        stats().ms_scan_kernel = ms_scan_kernel;
        stats().n_dropped = hs.n_dropped;
        stats().n_truncated = hs.n_truncated;
        return TFBS_OK;
    }
};

}  // namespace
