// host_common.hpp -- the context behind the C ABI: device / pinned buffers, a block on the device, the two slots of blocks in flight, the two lanes they run on
// Host side of libtfbs_b200.so (tfbs.cu is the map); one translation unit.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "kernels.cuh"

using namespace tfbs;

namespace {

thread_local std::string g_create_error;

// Buffers grow with some slack so that a slightly larger next block does not reallocate; the sanitizer build of tests/cuda_emu sets
// the slack to zero so that every out-of-bounds access is caught.
#ifndef TFBS_ALLOC_SLACK
#define TFBS_ALLOC_SLACK(bytes) ((bytes) / 8 + 256)
#endif

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    ~DevBuf() { if (p) cudaFree(p); }
    bool fits(size_t bytes) const { return bytes <= cap; }
    cudaError_t reserve(size_t bytes) {  // the caller makes sure no enqueued work still uses the old allocation (tfbs_ctx::grow)
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + TFBS_ALLOC_SLACK(bytes);
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct HostBuf {  // pinned; owned (cudaMallocHost) or bound to a piece of the caller's result arena
    void* p = nullptr;
    size_t cap = 0;
    bool owned = true;
    ~HostBuf() { if (p && owned) cudaFreeHost(p); }
    void bind(void* q, size_t bytes) {
        if (p && owned) cudaFreeHost(p);
        p = q;
        cap = bytes;
        owned = false;
    }
    cudaError_t reserve(size_t bytes, bool keep) {
        if (!owned) { p = nullptr; cap = 0; owned = true; }  // leave the arena: back to an own allocation
        if (bytes <= cap) return cudaSuccess;
        void* np = nullptr;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMallocHost(&np, want);
        if (e != cudaSuccess) return e;
        if (keep && p && cap) memcpy(np, p, cap);
        if (p) cudaFreeHost(p);
        p = np;
        cap = want;
        return cudaSuccess;
    }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// A block on the device: the caller's arrays plus host copies of the small per-region ones (planning, error messages).
struct BlockDev {
    bool valid = false;
    uint32_t R = 0, S = 0, H = 0, pitch = 0;
    uint64_t n_ref_bytes = 0, n_allele_bytes = 0, n_var = 0, n_inner = 0, n_carrier_rows = 0;
    DevBuf d_region_start, d_region_end, d_ref_off, d_ref_ascii, d_inner_off, d_inner, d_var_off, d_variants, d_allele_ascii, d_carriers;
    std::vector<int64_t> h_region_start, h_region_end;
    std::vector<uint64_t> h_ref_off;
    std::vector<uint32_t> h_inner_off, h_var_off;
    std::vector<uint64_t> h_ins_extra;  // per region: sum over variants of max(0, alt_len - 1)
    uint64_t h2d_bytes = 0;
};

// What a finished run exposes to tfbs_collect / tfbs_collect_grouped (pinned host memory).
struct Results {
    uint64_t n_rows = 0;
    HostBuf h_region, h_inner, h_pid, h_vmin, h_vmax;
    // dense: the reference's (left, right) vectors
    HostBuf h_left, h_right;
    uint32_t row_bytes = 4;
    bool have_dense = false;
    // grouped
    HostBuf h_base, h_bits, h_off, h_packed, h_ngroups, h_hg;
    uint64_t packed_words = 0;
    uint32_t hg_bytes = 4;
    bool have_grouped = false;
    // attribution (option "attribution", tfbs_get_attribution)
    HostBuf h_a_ref, h_a_toff, h_a_tcfg, h_a_tdiff, h_a_creg, h_a_cflags, h_a_croff, h_a_crec, h_a_goff, h_a_gcfg;
    bool have_attribution = false;
};

// Capacities a run of the configuration path was enqueued with (see DevPlan): sizes that only the device learns.
struct Caps {
    uint64_t seq = 0, d = 0, cfg = 0, vd = 0, items = 0, units = 0, dwords = 0, rows = 0, rowwords = 0;
    uint32_t capr = 0, groups = 0;
    uint64_t terms = 0;  // option "attribution": non-zero (row, configuration) differences
};

struct Slot {
    int state = 0;  // 0 free, 1 enqueued (nothing has been waited for), 2 finished (results final)
    bool full_mode = false;
    int lane = 0;   // tfbs_ctx::lane the block runs on (start_block)
    BlockDev own;
    BlockDev* in = nullptr;
    // device results of the configuration path: they outlive the shared scratch, which the next block reuses at once
    DevBuf d_status, d_plan, d_hap_group, d_gbase, d_hg_narrow;
    DevBuf d_o_region, d_o_inner, d_o_pid, d_o_vmin, d_o_vmax, d_o_base, d_o_bits, d_o_off, d_o_packed, d_left, d_right;
    DevBuf d_a_ref, d_a_toff, d_a_tcfg, d_a_tdiff, d_a_creg, d_a_cflags, d_a_croff, d_a_crec, d_a_goff, d_a_gcfg;  // attribution
    HostBuf h_status, h_plan;
    Results res;
    Caps caps;
    uint64_t seed = 0;
    uint64_t n_keys = 0;
    int rows_mode = 0;
    int attempts = 0;
    cudaEvent_t ev_in = nullptr, ev_done = nullptr, ev_t[8]{};
    tfbs_stats stats{};
    uint32_t fan_groups_cap = 0, fan_ctas = 0, fan_in_device_memory = 0;  // the fan-out of the last run (tfbs_fanout_info)
    bool attribution = false;                        // the run enqueued the attribution launches
    uint64_t att_cfgs = 0, att_seqs = 0, att_terms = 0;  // their sizes (configurations, distinct haplotypes, terms)
};

// The streams a block's work is enqueued on and the scratch its kernels share with the blocks before and after it on the same lane.
// Every block runs on lane 0 unless option "dual_stream" gives slot 1 a lane of its own (start_block): the kernels of consecutive
// blocks then overlap on the device instead of queueing on one stream.
struct Lane {
    cudaStream_t stream = nullptr;      // kernels
    cudaStream_t stream_in = nullptr;   // host -> device copies of the next block
    cudaStream_t stream_out = nullptr;  // device -> host copies of finished rows

    // scratch shared by consecutive blocks of the lane (their kernels are serialised on `stream`)
    DevBuf d_ref_codes, d_allele_codes, d_var_class, d_var_inwin, d_var_althash, d_ref_prefix;
    DevBuf d_sig, d_nd_in, d_leader, d_hap_group, d_ngroups, d_sum_nd, d_ref_used;
    DevBuf d_keys, d_vals, d_scanwork;
    DevBuf d_kbase, d_hap_mask, d_mask_base, d_region_dups, d_var_row;
    // distinct haplotypes ("sequences")
    DevBuf d_seq_region, d_seq_leader, d_seq_nd, d_seq_doff, d_dlist, d_segs, d_seq_nseg, d_seq_len, d_seq_hash, d_seq_flags, d_seq_ntake,
        d_seq_nitems, d_item_off, d_items, d_list, d_ent_units, d_ent_uoff, d_pk, d_nm, d_refhits, d_refcnt;
    // configuration path
    DevBuf d_var_cluster, d_var_sorted, d_ncfg, d_cfgbase, d_dwords, d_dbase, d_run_len, d_run_key, d_run_rep, d_run_cfg, d_cfg_src,
        d_cfg_net, d_mcount, d_moff, d_mfill, d_members, d_D, d_C0;
    DevBuf d_vq_region, d_vq_leader, d_vq_nd, d_vq_doff, d_vq_dlist, d_vq_segs, d_vq_nseg, d_vq_len, d_vq_flags, d_vq_ntake, d_vq_nitems,
        d_vq_item_off;
    DevBuf d_vmin, d_vmax, d_flag, d_rowwords, d_kbits, d_rowidx, d_rowoff;
    DevBuf d_fan_vec;  // k_fanout<true>: one count vector per CTA
    DevBuf d_att_eflag, d_att_cfgid, d_att_nrec, d_att_col, d_att_gn, d_att_tcnt;  // option "attribution"
    // full-scan path (lane 0 only)
    DevBuf d_gbase, d_cbase, d_C;
    DevBuf d_rows_region, d_rows_inner, d_rows_pid, d_rows_vmin, d_rows_vmax, d_rows_left, d_rows_right;
    DevBuf d_m_region, d_m_pattern, d_m_group, d_m_start;
    DevBuf d_hap_flags;
};

}  // namespace

struct tfbs_ctx {
    int device = 0;
    Lane lane[2];
    cudaDeviceProp prop{};
    std::string err;

    // options
    int rows_mode = TFBS_ROWS_VARYING;
    int record_matches = 0;
    uint64_t max_matches = 1u << 22;
    int verify_groups = 1;
    int scan_format = 0;
    uint64_t scratch_bytes = 24ull << 30;
    uint32_t table_budget = 160 * 1024;  // measured on configs[2] (802 patterns): 96 KB -> 5 chunk launches, 0.763 of the roof; 160 KB -> 3, 0.796
    int scan_ctas_per_sm = 0;  // < 0: fixed grid size (debugging)
    int delta = 1;             // 1: configuration path (delta scoring); 0: every distinct haplotype scored in full
    int64_t refhit_cap_opt = 0; // testing: reference hits kept per region (0 = automatic)
    int rows_width = 32;        // 32: counts are returned as u32; 0: narrowest of u8 / u16 / u32 that holds every count of the block
    int audit = 0;              // set by tfbs_audit_block: per-haplotype flags are kept
    int64_t tiny_caps = 0;      // testing: start the configuration path with minimal scratch so that every growth path runs
    int64_t test_reseed = 0;    // testing: the first attempt of every block is treated as a hash collision (repeated with another seed)
    int fan_vector = 0;         // 0: the fan-out's count vectors live in shared memory unless a region has too many groups; 1: always in device memory (testing)
    int attribution = 0;        // 1: the default path keeps the per-row configuration differences (tfbs_get_attribution)
    int dual_stream = 0;        // 1: a block in slot 1 of the default path runs on lane 1
    // attribution of the block the last tfbs_collect / tfbs_collect_grouped returned, copied to the host by that collect
    enum { ATT_NONE = 0, ATT_OFF, ATT_FULL_SCAN, ATT_READY };
    int att_state = ATT_NONE;
    tfbs_attribution att{};

    // patterns
    bool have_patterns = false;
    std::vector<tfbs_pattern> orig_patterns;          // the caller's list (tfbs_audit_block re-compiles it with lowered thresholds)
    std::vector<std::vector<int32_t>> orig_weights;
    CompiledPatterns cp;
    DevBuf d_table, d_chunks, d_runs, d_trip_pat, d_pat_len, d_pat_pid, d_pid_list;
    DevPatterns dpat{};

    // blocks in flight: a ring of two slots, plus the resident block of tfbs_upload_block
    Slot slot[2];
    int head = 0, in_flight = 0;   // oldest slot in flight, number of slots in flight
    int last = -1;                 // slot of the most recent tfbs_collect (stats, matches)
    BlockDev resident;
    BlockDev* last_block = nullptr;  // block of the most recent submit / upload (tfbs_audit_block)
    Caps hint;                     // largest needs seen so far (+ 25 %): what the next block is given
    uint8_t* arena = nullptr;      // tfbs_set_result_arena: grouped rows are copied straight into the caller's memory
    size_t arena_bytes = 0;

    // full-scan path
    std::vector<uint32_t> h_ngroups, h_sum_nd;
    std::vector<uint64_t> h_gbase, h_cbase, h_kbase;
    HostBuf h_m_region, h_m_pattern, h_m_group, h_m_start, h_hap_group;
    HostBuf h_totals;
    HostBuf h_hap_flags;
    std::vector<uint32_t> tie_region, tie_pattern, tie_group;  // tfbs_audit_block
    std::vector<int64_t> tie_start;
    uint64_t n_matches = 0;
    uint64_t n_matches_found = 0;  // hits the last run produced, also those that did not fit into the match buffer
    bool matches_truncated = false;

    cudaEvent_t ev[10]{};
};

namespace {

#define CK(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess) {                                                                              \
            ctx->err = std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " #call;                   \
            return TFBS_ERR_CUDA;                                                                             \
        }                                                                                                     \
    } while (0)

int fail(tfbs_ctx* ctx, int code, const std::string& msg) {
    ctx->err = msg;
    return code;
}

// Everything enqueued so far has finished (needed before an allocation that enqueued work may still use is replaced).
int quiesce(tfbs_ctx* ctx) {
    for (const Lane& L : ctx->lane) {
        CK(cudaStreamSynchronize(L.stream_in));
        CK(cudaStreamSynchronize(L.stream));
        CK(cudaStreamSynchronize(L.stream_out));
    }
    return TFBS_OK;
}

// Grow a device buffer that work in flight may still be using.
int grow(tfbs_ctx* ctx, DevBuf& buf, size_t bytes) {
    if (buf.fits(bytes)) return TFBS_OK;
    int rc = quiesce(ctx);
    if (rc) return rc;
    CK(buf.reserve(bytes));
    return TFBS_OK;
}

template <class T>
int upload_on(tfbs_ctx* ctx, cudaStream_t st, DevBuf& buf, const T* src, size_t n, uint64_t* bytes) {
    int rc = grow(ctx, buf, std::max<size_t>(1, n) * sizeof(T));
    if (rc) return rc;
    if (n) CK(cudaMemcpyAsync(buf.p, src, n * sizeof(T), cudaMemcpyHostToDevice, st));
    if (bytes) *bytes += n * sizeof(T);
    return TFBS_OK;
}

inline unsigned grid_for(uint64_t n, unsigned block) { return (unsigned)std::min<uint64_t>(0x7fffffffu, std::max<uint64_t>(1, (n + block - 1) / block)); }

// Shape of the block: everything that is read on the host to size the copies.
int validate_regions(tfbs_ctx* ctx, const tfbs_block* b) {
    if (!b) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "block is NULL");
    if (b->n_regions && (!b->region_start || !b->region_end || !b->ref_off || !b->inner_off || !b->var_off))
        return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "block has NULL region arrays");
    if ((uint64_t)b->n_samples * 2 > 0x7fffffffull) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "too many samples");
    uint32_t H = 2 * b->n_samples;
    if (b->n_carrier_rows && b->carrier_pitch < (H + 31) / 32) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "carrier_pitch is too small");
    for (uint32_t r = 0; r < b->n_regions; ++r) {
        if (b->region_start[r] < 0 || b->region_end[r] < b->region_start[r])
            return fail(ctx, TFBS_ERR_INVALID_ARGUMENT,
                        "region " + std::to_string(r) + " has an invalid extended window (main.rs:407 underflow)");
        if (b->region_end[r] - b->region_start[r] >= (1ll << 26))
            return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "region " + std::to_string(r) + " is longer than 2^26 bases");
        if (b->ref_off[r + 1] < b->ref_off[r] ||
            b->ref_off[r + 1] - b->ref_off[r] > (uint64_t)(b->region_end[r] - b->region_start[r] + 1))
            return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "region " + std::to_string(r) + ": reference window longer than the region");
        if (b->inner_off[r + 1] < b->inner_off[r] || b->var_off[r + 1] < b->var_off[r])
            return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "offset arrays must be non-decreasing");
    }
    return TFBS_OK;
}

// The records: allele ranges and carrier rows (what the kernels index with), and per region the bases insertions can add.
// Runs while the copies of the block are in flight.
int validate_variants(tfbs_ctx* ctx, const tfbs_block* b, BlockDev* B) {
    B->h_ins_extra.assign(b->n_regions, 0);
    for (uint32_t r = 0; r < b->n_regions; ++r)
        for (uint32_t v = b->var_off[r]; v < b->var_off[r + 1]; ++v) {
            const tfbs_variant& x = b->variants[v];
            if (x.ref_len == 0 || x.alt_len == 0) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "variant " + std::to_string(v) + " has an empty allele");
            if ((uint64_t)x.ref_off + x.ref_len > b->allele_bytes || (uint64_t)x.alt_off + x.alt_len > b->allele_bytes)
                return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "variant " + std::to_string(v) + " points outside allele_bases");
            if (x.carrier_row >= b->n_carrier_rows) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "variant " + std::to_string(v) + " has no carrier row");
            if (x.alt_len > 1) B->h_ins_extra[r] += x.alt_len - 1;
        }
    return TFBS_OK;
}

// Copies of the block are enqueued on `st`; the per-record checks run on the host while they are in flight.
int upload_block(tfbs_ctx* ctx, const tfbs_block* b, BlockDev* B, cudaStream_t st) {
    B->valid = false;
    int rc = validate_regions(ctx, b);
    if (rc) return rc;
    B->R = b->n_regions;
    B->S = b->n_samples;
    B->H = 2 * b->n_samples;
    B->pitch = b->carrier_pitch;
    const uint32_t R = B->R;
    B->n_ref_bytes = R ? b->ref_off[R] : 0;
    B->n_inner = R ? b->inner_off[R] : 0;
    B->n_var = R ? b->var_off[R] : 0;
    B->n_allele_bytes = b->allele_bytes;
    B->n_carrier_rows = b->n_carrier_rows;
    B->h_region_start.assign(b->region_start, b->region_start + R);
    B->h_region_end.assign(b->region_end, b->region_end + R);
    if (R) {
        B->h_ref_off.assign(b->ref_off, b->ref_off + R + 1);
        B->h_inner_off.assign(b->inner_off, b->inner_off + R + 1);
        B->h_var_off.assign(b->var_off, b->var_off + R + 1);
    } else {
        B->h_ref_off.assign(1, 0);
        B->h_inner_off.assign(1, 0);
        B->h_var_off.assign(1, 0);
    }
    if (R && B->n_var && !b->variants) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "block has records but variants is NULL");
    B->h2d_bytes = 0;
    uint64_t* nb = &B->h2d_bytes;
    if ((rc = upload_on(ctx, st, B->d_region_start, b->region_start, R, nb))) return rc;
    if ((rc = upload_on(ctx, st, B->d_region_end, b->region_end, R, nb))) return rc;
    if ((rc = upload_on(ctx, st, B->d_ref_off, B->h_ref_off.data(), R + 1, nb))) return rc;
    if ((rc = upload_on(ctx, st, B->d_ref_ascii, b->ref_bases, B->n_ref_bytes, nb))) return rc;
    if ((rc = upload_on(ctx, st, B->d_inner_off, B->h_inner_off.data(), R + 1, nb))) return rc;
    if ((rc = upload_on(ctx, st, B->d_inner, b->inner, B->n_inner, nb))) return rc;
    if ((rc = upload_on(ctx, st, B->d_var_off, B->h_var_off.data(), R + 1, nb))) return rc;
    if ((rc = upload_on(ctx, st, B->d_variants, b->variants, B->n_var, nb))) return rc;
    if ((rc = upload_on(ctx, st, B->d_allele_ascii, b->allele_bases, B->n_allele_bytes, nb))) return rc;
    if ((rc = upload_on(ctx, st, B->d_carriers, b->carriers, (size_t)B->n_carrier_rows * B->pitch, nb))) return rc;
    // the per-record checks overlap the copies (asynchronous when the caller's buffers are page-locked); no kernel has been enqueued yet
    if ((rc = validate_variants(ctx, b, B))) {
        cudaStreamSynchronize(st);
        return rc;
    }
    B->valid = true;
    return TFBS_OK;
}

// Scratch the input encoding of a block needs (shared by both pipelines).
int reserve_encoding(tfbs_ctx* ctx, Lane& L, const BlockDev& B) {
    int rc;
    if ((rc = grow(ctx, L.d_ref_codes, std::max<uint64_t>(1, B.n_ref_bytes)))) return rc;
    if ((rc = grow(ctx, L.d_allele_codes, std::max<uint64_t>(1, B.n_allele_bytes)))) return rc;
    if ((rc = grow(ctx, L.d_var_class, std::max<uint64_t>(1, B.n_var) * 4))) return rc;
    if ((rc = grow(ctx, L.d_var_inwin, std::max<uint64_t>(1, B.n_var)))) return rc;
    if ((rc = grow(ctx, L.d_var_althash, std::max<uint64_t>(1, B.n_var) * 8))) return rc;
    if ((rc = grow(ctx, L.d_ref_prefix, (B.n_ref_bytes + B.R + 1) * 8))) return rc;
    return TFBS_OK;
}

// The block's arrays are only read: both lanes may run the resident block at once.  Its encoding is the lane's scratch.
DevBlock dev_block(const Lane& L, const BlockDev& B) {
    DevBlock b{};
    b.R = B.R;
    b.S = B.S;
    b.H = B.H;
    b.region_start = B.d_region_start.as<i64>();
    b.region_end = B.d_region_end.as<i64>();
    b.ref_off = B.d_ref_off.as<u64>();
    b.ref_codes = L.d_ref_codes.as<u8>();
    b.inner_off = B.d_inner_off.as<u32>();
    b.inner = B.d_inner.as<tfbs_inner_region>();
    b.var_off = B.d_var_off.as<u32>();
    b.variants = B.d_variants.as<tfbs_variant>();
    b.allele_codes = L.d_allele_codes.as<u8>();
    b.carriers = B.d_carriers.as<u32>();
    b.pitch = B.pitch;
    b.var_class = L.d_var_class.as<u32>();
    b.var_inwin = L.d_var_inwin.as<u8>();
    b.var_althash = L.d_var_althash.as<u64>();
    b.ref_prefix = L.d_ref_prefix.as<u64>();
    return b;
}

// exclusive scan of d_in[0, n) into d_out[0, n], total into d_out[n]; n = n_ptr ? min(*n_ptr, n_cap) : n_cap (one launch)
int device_scan(tfbs_ctx* ctx, Lane& L, const uint32_t* d_in, uint64_t n_cap, const u64* n_ptr, u64* d_out, uint32_t* launches) {
    cudaStream_t st = L.stream;
    const uint64_t tiles = (n_cap + SCAN_TILE - 1) / SCAN_TILE;
    if (tiles == 0) {
        CK(cudaMemsetAsync(d_out, 0, sizeof(u64), st));
        return TFBS_OK;
    }
    if (!L.d_scanwork.fits((tiles + 1) * 8)) {
        int rc = grow(ctx, L.d_scanwork, (tiles + 1) * 8);
        if (rc) return rc;
    }
    CK(cudaMemsetAsync(L.d_scanwork.p, 0, (tiles + 1) * 8, st));
    TFBS_LAUNCH(k_exclusive_scan, (unsigned)tiles, SCAN_THREADS, 0, st)(d_in, n_cap, n_ptr, d_out, L.d_scanwork.as<u64>());
    if (launches) ++*launches;
    CK(cudaGetLastError());
    return TFBS_OK;
}

}  // namespace
