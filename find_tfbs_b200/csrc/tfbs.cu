// tfbs.cu -- C ABI (include/tfbs.h) over the sm_100a kernels in kernels.cuh.
//
//   host_common.hpp      the context: device / pinned buffers, a block on the device, two slots of blocks in flight, two lanes of
//                        streams and scratch
//   pipeline_config.hpp  the default path: configurations + fan-out into grouped rows, enqueued without a single host round trip
//   pipeline_full.hpp    every distinct haplotype scored in full like the reference ("delta" = 0, the hit list, the audit)
//
// One context = one CUDA device.  tfbs_submit_block copies a block on the copy-in stream of its lane and enqueues its kernels on the
// lane's kernel stream; tfbs_collect waits for the oldest block, fetches its rows on the lane's copy-out stream and is the only place
// the host waits.
// There is no CPU fallback: every entry point that computes fails with TFBS_ERR_CUDA when no device is usable.
#include "host_common.hpp"
#include "pipeline_config.hpp"
#include "pipeline_full.hpp"

namespace {

bool wants_full(const tfbs_ctx* ctx) { return !ctx->delta || ctx->record_matches || ctx->audit; }

// Run (full path) or enqueue (configuration path) a block on the next free slot: the block `in` that is on the device already, or
// (in == NULL) the caller's block `b`, copied into the slot first.
int start_block(tfbs_ctx* ctx, BlockDev* in, const tfbs_block* b) {
    if (!ctx->have_patterns) return fail(ctx, TFBS_ERR_STATE, "tfbs_set_patterns has not been called");
    if (ctx->in_flight >= 2) return fail(ctx, TFBS_ERR_STATE, "two blocks are already in flight on this context: call tfbs_collect first");
    if (ctx->sites && !ctx->attribution)
        return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "option sites needs option attribution = 1: sites refer to its configuration ids");
    const int k = (ctx->head + ctx->in_flight) % 2;
    Slot* slot = &ctx->slot[k];
    slot->lane = ctx->dual_stream && !wants_full(ctx) ? k : 0;  // option "dual_stream": consecutive blocks run on different lanes
    Lane& L = ctx->lane[slot->lane];
    const bool copies_pending = !in;
    int rc;
    if (copies_pending) {
        if ((rc = upload_block(ctx, b, &slot->own, L.stream_in))) return rc;
        in = &slot->own;
    }
    if (!in->valid) return fail(ctx, TFBS_ERR_STATE, "no block has been uploaded");
    slot->in = in;
    slot->state = 0;
    CK(cudaEventRecord(slot->ev_in, copies_pending ? L.stream_in : L.stream));
    if (wants_full(ctx)) {
        if (ctx->in_flight) return fail(ctx, TFBS_ERR_STATE, "the full scan (delta = 0, record_matches, audit) runs one block at a time: call tfbs_collect first");
        CK(cudaStreamWaitEvent(L.stream, slot->ev_in, 0));
        slot->full_mode = true;
        rc = FullPipeline(ctx, slot).run();
        if (rc) return rc;
        slot->state = 2;
    } else {
        rc = ConfigPipeline(ctx, slot).enqueue(true);
        if (rc) return rc;
    }
    ++ctx->in_flight;
    ctx->last_block = in;
    return TFBS_OK;
}

// Oldest block in flight: wait for it, make its results final.
int finish_oldest(tfbs_ctx* ctx, Slot** out) {
    if (!ctx->in_flight) return fail(ctx, TFBS_ERR_STATE, "tfbs_collect called without a block in flight (tfbs_submit_block / tfbs_run_resident first)");
    Slot* slot = &ctx->slot[ctx->head];
    if (slot->state == 1) {
        int rc = ConfigPipeline(ctx, slot).finalize();
        if (rc) {  // the block is lost; the context stays usable
            slot->state = 0;
            ctx->head = (ctx->head + 1) % 2;
            --ctx->in_flight;
            return rc;
        }
    }
    *out = slot;
    return TFBS_OK;
}

// The collect that returns a block also brings its attribution, sites and record sites to the host (options "attribution", "sites",
// "record_sites"): a later block may take the slot's device buffers before tfbs_get_attribution is called.
int take_attribution(tfbs_ctx* ctx, Slot* slot) {
    if (slot->full_mode) { ctx->att_state = ctx->site_state = ctx->rec_state = tfbs_ctx::ATT_FULL_SCAN; return TFBS_OK; }
    ctx->att_state = ctx->site_state = ctx->rec_state = tfbs_ctx::ATT_OFF;
    int rc;
    if (slot->attribution) {
        if ((rc = ConfigPipeline(ctx, slot).fetch_attribution())) return rc;
        if (slot->sites) {
            if ((rc = ConfigPipeline(ctx, slot).fetch_sites())) return rc;
            const Results& res = slot->res;
            tfbs_sites& so = ctx->site;
            so.n_cfgs = slot->att_cfgs;
            so.site_off = res.h_s_off.as<uint64_t>();
            so.pattern_index = res.h_s_pat.as<uint32_t>();
            so.start = res.h_s_start.as<int64_t>();
            so.score = res.h_s_score.as<int32_t>();
            so.change = res.h_s_change.as<int8_t>();
            ctx->site_state = tfbs_ctx::ATT_READY;
        }
        const Results& res = slot->res;
        tfbs_attribution& out = ctx->att;
        memset(&out, 0, sizeof out);
        out.n_rows = res.n_rows;
        out.ref_count = res.h_a_ref.as<uint32_t>();
        out.term_off = res.h_a_toff.as<uint64_t>();
        out.term_cfg = res.h_a_tcfg.as<uint32_t>();
        out.term_diff = res.h_a_tdiff.as<int32_t>();
        out.n_cfgs = slot->att_cfgs;
        out.cfg_region = res.h_a_creg.as<uint32_t>();
        out.cfg_flags = res.h_a_cflags.as<uint8_t>();
        out.cfg_rec_off = res.h_a_croff.as<uint64_t>();
        out.cfg_rec = res.h_a_crec.as<uint32_t>();
        out.n_groups_total = slot->att_seqs;
        out.group_cfg_off = res.h_a_goff.as<uint64_t>();
        out.group_cfg = res.h_a_gcfg.as<uint32_t>();
        ctx->att_state = tfbs_ctx::ATT_READY;
    }
    if (slot->record_sites) {
        if ((rc = ConfigPipeline(ctx, slot).fetch_record_sites())) return rc;
        const Results& res = slot->res;
        tfbs_record_sites& ro = ctx->rec;
        ro.n_records = slot->n_records;
        ro.rec_flags = res.h_r_flags.as<uint8_t>();
        ro.site_off = res.h_r_off.as<uint64_t>();
        ro.pattern_index = res.h_r_pat.as<uint32_t>();
        ro.start = res.h_r_start.as<int64_t>();
        ro.score = res.h_r_score.as<int32_t>();
        ro.change = res.h_r_change.as<int8_t>();
        ctx->rec_state = tfbs_ctx::ATT_READY;
    }
    return TFBS_OK;
}

void retire_oldest(tfbs_ctx* ctx) {
    ctx->last = ctx->head;
    ctx->slot[ctx->head].state = 0;
    ctx->head = (ctx->head + 1) % 2;
    --ctx->in_flight;
}

// Compile the pattern list into scan tables and upload them.
int install_patterns(tfbs_ctx* ctx, const tfbs_pattern* patterns, uint32_t n_patterns) {
    CK(cudaSetDevice(ctx->device));
    ctx->have_patterns = false;
    if (n_patterns == 0) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "assertion failed: pwm_list.len() > 0");  // main.rs:238
    int rc = quiesce(ctx);  // blocks in flight still read the old tables
    if (rc) return rc;
    size_t max_smem = ctx->prop.sharedMemPerBlockOptin;
    size_t fixed = sizeof(CtaShared) + SCAN_WARPS * sizeof(WarpShared) + 1024;
    uint32_t budget = (uint32_t)std::min<size_t>(ctx->table_budget, max_smem > fixed ? max_smem - fixed : 0);
    std::string err;
    CompiledPatterns cp;
    rc = compile_patterns(patterns, n_patterns, budget, ctx->scan_format == 1, &cp, &err);
    if (rc != TFBS_OK) return fail(ctx, rc, err);
    ctx->cp = std::move(cp);
    const CompiledPatterns& c = ctx->cp;
    std::vector<uint64_t> table = c.table;
    table.resize(table.size() + 2, 0);  // 128-bit loads may read one word past the end
    cudaStream_t st = ctx->lane[0].stream;
    if ((rc = upload_on(ctx, st, ctx->d_table, table.data(), table.size(), nullptr))) return rc;
    if ((rc = upload_on(ctx, st, ctx->d_chunks, c.chunks.data(), c.chunks.size(), nullptr))) return rc;
    if ((rc = upload_on(ctx, st, ctx->d_runs, c.runs.data(), c.runs.size(), nullptr))) return rc;
    if ((rc = upload_on(ctx, st, ctx->d_trip_pat, c.trip_pat.data(), c.trip_pat.size(), nullptr))) return rc;
    if ((rc = upload_on(ctx, st, ctx->d_pat_len, c.pat_len.data(), c.pat_len.size(), nullptr))) return rc;
    if ((rc = upload_on(ctx, st, ctx->d_pat_pid, c.pat_pid_index.data(), c.pat_pid_index.size(), nullptr))) return rc;
    if ((rc = upload_on(ctx, st, ctx->d_pat_w, c.pat_w.data(), c.pat_w.size(), nullptr))) return rc;
    if ((rc = upload_on(ctx, st, ctx->d_pid_list, c.pid_list.data(), c.pid_list.size(), nullptr))) return rc;
    CK(cudaStreamSynchronize(st));
    DevPatterns& d = ctx->dpat;
    d.table = ctx->d_table.as<u64>();
    d.chunks = ctx->d_chunks.as<ChunkDesc>();
    d.runs = ctx->d_runs.as<RunDesc>();
    d.trip_pat = ctx->d_trip_pat.as<int>();
    d.pat_len = ctx->d_pat_len.as<u32>();
    d.pat_pid_index = ctx->d_pat_pid.as<u32>();
    d.pat_w = ctx->d_pat_w.as<int>();
    d.n_chunks = (u32)c.chunks.size();
    d.n_pid = (u32)c.pid_list.size();
    d.n_patterns = (u32)c.patterns.size();
    d.max_len = c.max_len;
    d.sum_len = c.sum_len;
    d.sum_len_sq = c.sum_len_sq;
    ctx->have_patterns = true;
    return TFBS_OK;
}

// Drop every block in flight (after a failed call, before a mode that owns the device).
int drain(tfbs_ctx* ctx) {
    int rc = quiesce(ctx);
    ctx->slot[0].state = ctx->slot[1].state = 0;
    ctx->in_flight = 0;
    ctx->head = 0;
    return rc;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------------
extern "C" {

int tfbs_abi_version(void) { return TFBS_ABI_VERSION; }

int tfbs_create(int device, tfbs_ctx** out) {
    if (!out) return TFBS_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        g_create_error = std::string("no usable CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                         " (this library has no CPU fallback)";
        return TFBS_ERR_CUDA;
    }
    if (device < 0 || device >= n) {
        g_create_error = "device index out of range";
        return TFBS_ERR_INVALID_ARGUMENT;
    }
    if ((e = cudaSetDevice(device)) != cudaSuccess) {
        g_create_error = std::string("cudaSetDevice failed: ") + cudaGetErrorString(e);
        return TFBS_ERR_CUDA;
    }
    tfbs_ctx* ctx = new tfbs_ctx();
    ctx->device = device;
    e = cudaGetDeviceProperties(&ctx->prop, device);
    for (Lane& L : ctx->lane)
        for (cudaStream_t* s : {&L.stream, &L.stream_in, &L.stream_out})
            if (e == cudaSuccess) e = cudaStreamCreateWithFlags(s, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        g_create_error = std::string("CUDA initialisation failed: ") + cudaGetErrorString(e);
        tfbs_destroy(ctx);
        return TFBS_ERR_CUDA;
    }
    if (ctx->prop.major < 10) {
        g_create_error = std::string("device ") + ctx->prop.name + " is not sm_100-class; this library carries sm_100a code only";
        tfbs_destroy(ctx);
        return TFBS_ERR_CUDA;
    }
    for (auto& ev : ctx->ev) cudaEventCreate(&ev);
    for (Slot& s : ctx->slot) {
        cudaEventCreate(&s.ev_in);
        cudaEventCreate(&s.ev_done);
        for (auto& ev : s.ev_t) cudaEventCreate(&ev);
    }
    // every pipeline reads its table; lane 1's streams are not ordered after lane 0's, so the table is complete before the call returns
    TFBS_LAUNCH(k_hash_pow_init, 1, 32, 0, ctx->lane[0].stream)();
    if ((e = cudaGetLastError()) != cudaSuccess || (e = cudaStreamSynchronize(ctx->lane[0].stream)) != cudaSuccess) {
        g_create_error = std::string("CUDA initialisation failed: ") + cudaGetErrorString(e);
        tfbs_destroy(ctx);
        return TFBS_ERR_CUDA;
    }
    *out = ctx;
    return TFBS_OK;
}

void tfbs_destroy(tfbs_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    for (Lane& L : ctx->lane)
        for (cudaStream_t s : {L.stream_in, L.stream, L.stream_out})
            if (s) cudaStreamSynchronize(s);
    for (auto& ev : ctx->ev)
        if (ev) cudaEventDestroy(ev);
    for (Slot& s : ctx->slot) {
        if (s.ev_in) cudaEventDestroy(s.ev_in);
        if (s.ev_done) cudaEventDestroy(s.ev_done);
        for (auto& ev : s.ev_t)
            if (ev) cudaEventDestroy(ev);
    }
    if (ctx->arena) cudaHostUnregister(ctx->arena);
    for (Lane& L : ctx->lane)
        for (cudaStream_t s : {L.stream, L.stream_in, L.stream_out})
            if (s) cudaStreamDestroy(s);
    delete ctx;
}

const char* tfbs_last_error(const tfbs_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int tfbs_set_option(tfbs_ctx* ctx, const char* key, int64_t value) {
    if (!ctx || !key) return TFBS_ERR_INVALID_ARGUMENT;
    std::string k(key);
    if (k == "rows_mode") {
        if (value != TFBS_ROWS_VARYING && value != TFBS_ROWS_ALL_KEYS) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "rows_mode must be 0 or 1");
        ctx->rows_mode = (int)value;
    } else if (k == "record_matches") ctx->record_matches = value != 0;
    else if (k == "max_matches") ctx->max_matches = (uint64_t)std::max<int64_t>(1, value);
    else if (k == "verify_groups") ctx->verify_groups = value != 0;
    else if (k == "scan_format") { ctx->scan_format = (int)value; ctx->have_patterns = false; }
    else if (k == "scratch_mb") ctx->scratch_bytes = (uint64_t)std::max<int64_t>(64, value) << 20;
    else if (k == "table_budget_kb") { ctx->table_budget = (uint32_t)std::max<int64_t>(8, value) * 1024; ctx->have_patterns = false; }
    else if (k == "scan_ctas_per_sm") ctx->scan_ctas_per_sm = (int)value;
    else if (k == "delta") ctx->delta = value != 0;
    else if (k == "refhit_cap") ctx->refhit_cap_opt = std::max<int64_t>(0, value);
    else if (k == "tiny_caps") ctx->tiny_caps = value;
    else if (k == "test_reseed") ctx->test_reseed = value;
    else if (k == "test_sig_bits") {
        if (value < 0 || value > 63) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "test_sig_bits must be 0 (off) .. 63");
        ctx->test_sig_bits = (int)value;
    }
    else if (k == "fan_vector") {
        if (value != 0 && value != 1) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "fan_vector must be 0 (automatic) or 1 (device memory)");
        ctx->fan_vector = (int)value;
    }
    else if (k == "region_tables") {
        if (value != 0 && value != 1) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "region_tables must be 0 or 1");
        ctx->region_tables = (int)value;
    }
    else if (k == "attribution") {
        if (value != 0 && value != 1) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "attribution must be 0 or 1");
        ctx->attribution = (int)value;
    }
    else if (k == "sites") {
        if (value != 0 && value != 1) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "sites must be 0 or 1");
        ctx->sites = (int)value;
    }
    else if (k == "record_sites") {
        if (value != 0 && value != 1) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "record_sites must be 0 or 1");
        ctx->record_sites = (int)value;
    }
    else if (k == "rows_width") {
        if (value != 0 && value != 32) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "rows_width must be 32 or 0 (automatic)");
        ctx->rows_width = (int)value;
    }
    else if (k == "dual_stream") {
        if (ctx->in_flight) return fail(ctx, TFBS_ERR_STATE, "dual_stream with blocks in flight: call tfbs_collect first");
        ctx->dual_stream = value != 0;
    }
    else return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "unknown option " + k);
    return TFBS_OK;
}

int tfbs_set_patterns(tfbs_ctx* ctx, const tfbs_pattern* patterns, uint32_t n_patterns) {
    if (!ctx || (!patterns && n_patterns)) return TFBS_ERR_INVALID_ARGUMENT;
    int rc = install_patterns(ctx, patterns, n_patterns);
    if (rc != TFBS_OK) return rc;
    // keep the caller's list: tfbs_audit_block compiles it a second time with every threshold lowered by one
    ctx->orig_patterns.assign(patterns, patterns + n_patterns);
    ctx->orig_weights.assign(n_patterns, std::vector<int32_t>());
    for (uint32_t i = 0; i < n_patterns; ++i)
        if (patterns[i].kind == TFBS_PATTERN_PWM && patterns[i].weights && patterns[i].len) {
            ctx->orig_weights[i].assign(patterns[i].weights, patterns[i].weights + 4 * (size_t)patterns[i].len);
            ctx->orig_patterns[i].weights = ctx->orig_weights[i].data();
        } else {
            ctx->orig_patterns[i].weights = nullptr;
        }
    return TFBS_OK;
}

int tfbs_upload_block(tfbs_ctx* ctx, const tfbs_block* block) {
    if (!ctx) return TFBS_ERR_INVALID_ARGUMENT;
    CK(cudaSetDevice(ctx->device));
    int rc = drain(ctx);  // the resident block may still be read by runs in flight
    if (rc) return rc;
    rc = upload_block(ctx, block, &ctx->resident, ctx->lane[0].stream_in);
    if (rc) return rc;
    CK(cudaStreamSynchronize(ctx->lane[0].stream_in));
    ctx->last_block = &ctx->resident;
    return TFBS_OK;
}

int tfbs_run_resident(tfbs_ctx* ctx) {
    if (!ctx) return TFBS_ERR_INVALID_ARGUMENT;
    CK(cudaSetDevice(ctx->device));
    if (!ctx->resident.valid) return fail(ctx, TFBS_ERR_STATE, "no block has been uploaded");
    return start_block(ctx, &ctx->resident, nullptr);
}

int tfbs_submit_block(tfbs_ctx* ctx, const tfbs_block* block) {
    if (!ctx) return TFBS_ERR_INVALID_ARGUMENT;
    CK(cudaSetDevice(ctx->device));
    return start_block(ctx, nullptr, block);
}

int tfbs_collect(tfbs_ctx* ctx, tfbs_rows* out) {
    if (!ctx || !out) return TFBS_ERR_INVALID_ARGUMENT;
    CK(cudaSetDevice(ctx->device));
    ctx->att_state = ctx->site_state = ctx->rec_state = tfbs_ctx::ATT_NONE;
    Slot* slot = nullptr;
    int rc = finish_oldest(ctx, &slot);
    if (rc) return rc;
    if (!slot->full_mode && (rc = ConfigPipeline(ctx, slot).fetch_dense())) { retire_oldest(ctx); return rc; }
    if ((rc = take_attribution(ctx, slot))) { retire_oldest(ctx); return rc; }
    const Results& res = slot->res;
    out->n_rows = res.n_rows;
    out->n_samples = slot->in->S;
    out->count_bytes = res.n_rows ? res.row_bytes : 4;
    out->region = res.h_region.as<uint32_t>();
    out->inner = res.h_inner.as<uint32_t>();
    out->pattern_id = res.h_pid.as<uint16_t>();
    out->vmin = res.h_vmin.as<uint32_t>();
    out->vmax = res.h_vmax.as<uint32_t>();
    out->left = res.h_left.as<uint32_t>();
    out->right = res.h_right.as<uint32_t>();
    retire_oldest(ctx);
    return TFBS_OK;
}

int tfbs_collect_grouped(tfbs_ctx* ctx, tfbs_grouped_rows* out) {
    if (!ctx || !out) return TFBS_ERR_INVALID_ARGUMENT;
    CK(cudaSetDevice(ctx->device));
    ctx->att_state = ctx->site_state = ctx->rec_state = tfbs_ctx::ATT_NONE;
    Slot* slot = nullptr;
    int rc = finish_oldest(ctx, &slot);
    if (rc) return rc;
    if (slot->full_mode) {
        ctx->att_state = ctx->site_state = ctx->rec_state = tfbs_ctx::ATT_FULL_SCAN;
        retire_oldest(ctx);
        return fail(ctx, TFBS_ERR_STATE, "grouped rows come from the default scoring mode (delta = 1, record_matches off): use tfbs_collect");
    }
    if ((rc = ConfigPipeline(ctx, slot).fetch_grouped()) || (rc = take_attribution(ctx, slot))) { retire_oldest(ctx); return rc; }
    const Results& res = slot->res;
    memset(out, 0, sizeof *out);
    out->n_rows = res.n_rows;
    out->n_samples = slot->in->S;
    out->n_regions = slot->in->R;
    out->region = res.h_region.as<uint32_t>();
    out->inner = res.h_inner.as<uint32_t>();
    out->pattern_id = res.h_pid.as<uint16_t>();
    out->vmin = res.h_vmin.as<uint32_t>();
    out->vmax = res.h_vmax.as<uint32_t>();
    out->base = res.h_base.as<uint32_t>();
    out->bits = res.h_bits.as<uint8_t>();
    out->offset = res.h_off.as<uint64_t>();
    out->packed = res.h_packed.as<uint32_t>();
    out->packed_words = res.packed_words;
    out->n_groups = res.h_ngroups.as<uint32_t>();
    out->hap_group = res.h_hg.p;
    out->hap_group_bytes = res.hg_bytes;
    retire_oldest(ctx);
    return TFBS_OK;
}

int tfbs_set_result_arena(tfbs_ctx* ctx, void* base, size_t bytes) {
    if (!ctx) return TFBS_ERR_INVALID_ARGUMENT;
    CK(cudaSetDevice(ctx->device));
    int rc = quiesce(ctx);
    if (rc) return rc;
    if (ctx->in_flight) return fail(ctx, TFBS_ERR_STATE, "tfbs_set_result_arena with blocks in flight: call tfbs_collect first");
    ctx->head = 0;  // a block's rows go to the half of its slot: the next block to the first half
    if (ctx->arena) {
        cudaHostUnregister(ctx->arena);
        for (Slot& s : ctx->slot)
            for (HostBuf* hb : {&s.res.h_region, &s.res.h_inner, &s.res.h_pid, &s.res.h_vmin, &s.res.h_vmax, &s.res.h_base, &s.res.h_bits, &s.res.h_off,
                                &s.res.h_packed, &s.res.h_ngroups, &s.res.h_hg})
                if (!hb->owned) hb->bind(nullptr, 0);
        ctx->arena = nullptr;
        ctx->arena_bytes = 0;
    }
    if (!base) return TFBS_OK;
    if (bytes < 2 * 4096 || ((uintptr_t)base & 63)) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "the result arena must be 64-byte aligned and hold at least 8 KB");
    CK(cudaHostRegister(base, bytes, cudaHostRegisterDefault));
    ctx->arena = (uint8_t*)base;
    ctx->arena_bytes = bytes;
    memset(base, 0, sizeof(tfbs_arena_header));
    memset((uint8_t*)base + bytes / 2, 0, sizeof(tfbs_arena_header));
    return TFBS_OK;
}

int tfbs_expand_rows(const tfbs_grouped_rows* g, uint64_t first_row, uint64_t n_rows, uint32_t* left, uint32_t* right) {
    if (!g || (n_rows && (!left || !right)) || first_row > g->n_rows || n_rows > g->n_rows - first_row) return TFBS_ERR_INVALID_ARGUMENT;
    const uint32_t S = g->n_samples;
    const uint64_t H = 2ull * S;
    for (uint64_t i = 0; i < n_rows; ++i) {
        const uint64_t row = first_row + i;
        const uint32_t r = g->region[row], base = g->base[row], bits = g->bits[row];
        if (r >= g->n_regions || (bits != 0 && bits != 1 && bits != 2 && bits != 4 && bits != 8 && bits != 16 && bits != 32)) return TFBS_ERR_INVALID_ARGUMENT;
        const uint32_t* pk = g->packed + g->offset[row];
        // bits is a power of two: entry g sits in word g >> (5 - log2 bits) at bit (g mod (32 / bits)) << log2 bits
        const uint32_t lb = bits ? (uint32_t)__builtin_ctz(bits) : 0, wshift = 5 - lb, per_mask = bits ? (32u >> lb) - 1 : 0;
        const uint32_t mask = bits == 32 ? 0xffffffffu : ((1u << bits) - 1);
        uint32_t* l = left + i * S;
        uint32_t* rt = right + i * S;
        auto count = [&](uint32_t grp) { return bits ? base + ((pk[grp >> wshift] >> ((grp & per_mask) << lb)) & mask) : base; };
        if (g->hap_group_bytes == 2) {
            const uint16_t* hg = (const uint16_t*)g->hap_group + (uint64_t)r * H;
            for (uint32_t s = 0; s < S; ++s) { l[s] = count(hg[2 * s]); rt[s] = count(hg[2 * s + 1]); }
        } else {
            const uint32_t* hg = (const uint32_t*)g->hap_group + (uint64_t)r * H;
            for (uint32_t s = 0; s < S; ++s) { l[s] = count(hg[2 * s]); rt[s] = count(hg[2 * s + 1]); }
        }
    }
    return TFBS_OK;
}

// Sample blocks (SURVEY 8e, BASELINE.json configs[3]): counts are per sample, so the rows of disjoint sample ranges concatenate along
// the sample axis, but the min != max filter of counts_as_genotypes (main.rs:450-458) needs every sample: it is applied here, after
// the gather, on the (vmin, vmax) of each block's TFBS_ROWS_ALL_KEYS rows.  A k-way merge over the rows' key order.
int tfbs_merge_sample_blocks(const tfbs_grouped_rows* const* parts, uint32_t n_parts, uint64_t cap, uint32_t* region, uint32_t* inner,
                             uint16_t* pattern_id, uint32_t* vmin, uint32_t* vmax, uint64_t* part_row, uint64_t* n_out) {
    if (!n_out || (n_parts && !parts) || (cap && (!region || !inner || !pattern_id || !vmin || !vmax || !part_row))) return TFBS_ERR_INVALID_ARGUMENT;
    for (uint32_t p = 0; p < n_parts; ++p)
        if (!parts[p]) return TFBS_ERR_INVALID_ARGUMENT;
    struct Key {
        uint32_t region, inner;
        uint16_t pid;
        bool operator<(const Key& o) const { return region != o.region ? region < o.region : (pid != o.pid ? pid < o.pid : inner < o.inner); }
        bool operator==(const Key& o) const { return region == o.region && pid == o.pid && inner == o.inner; }
    };
    auto key_at = [&](uint32_t p, uint64_t i) { return Key{parts[p]->region[i], parts[p]->inner[i], parts[p]->pattern_id[i]}; };
    std::vector<uint64_t> cur(n_parts, 0);
    uint64_t n = 0;
    for (;;) {
        bool any = false;
        Key k{};
        for (uint32_t p = 0; p < n_parts; ++p) {
            if (cur[p] >= parts[p]->n_rows) continue;
            const Key kp = key_at(p, cur[p]);
            if (cur[p] && !(key_at(p, cur[p] - 1) < kp)) return TFBS_ERR_INVALID_ARGUMENT;  // rows are not in key order
            if (!any || kp < k) k = kp;
            any = true;
        }
        if (!any) break;
        // a block without the key had no hit for it: all its samples count 0 (main.rs:517-528)
        uint32_t lo = 0xffffffffu, hi = 0;
        for (uint32_t p = 0; p < n_parts; ++p) {
            const bool has = cur[p] < parts[p]->n_rows && key_at(p, cur[p]) == k;
            const uint32_t a = has ? parts[p]->vmin[cur[p]] : 0u, b = has ? parts[p]->vmax[cur[p]] : 0u;
            lo = std::min(lo, a);
            hi = std::max(hi, b);
        }
        const bool keep = lo != hi;
        for (uint32_t p = 0; p < n_parts; ++p) {
            const bool has = cur[p] < parts[p]->n_rows && key_at(p, cur[p]) == k;
            if (keep && n < cap) part_row[(uint64_t)p * cap + n] = has ? cur[p] : ~0ull;
            if (has) ++cur[p];
        }
        if (keep) {
            if (n < cap) { region[n] = k.region; inner[n] = k.inner; pattern_id[n] = k.pid; vmin[n] = lo; vmax[n] = hi; }
            ++n;
        }
    }
    *n_out = n;
    return TFBS_OK;
}

// load_peak_files' merge (bed.rs:37-45 -> RangeStack, range.rs:43-87) on the device: stable rank by start, prefix maximum of the ends.
int tfbs_merge_regions(tfbs_ctx* ctx, const uint64_t* start, const uint64_t* end, uint64_t n, uint64_t* out_start, uint64_t* out_end, uint64_t* n_out) {
    if (!ctx || !n_out || (n && (!start || !end || !out_start || !out_end))) return TFBS_ERR_INVALID_ARGUMENT;
    *n_out = 0;
    if (n == 0) return TFBS_OK;
    if (n > 0x7fffffffull) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "too many ranges");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->lane[0].stream;
    DevBuf d_in, d_out, d_order, d_misc;
    CK(d_in.reserve(n * 16));
    CK(d_out.reserve(n * 16));
    CK(d_order.reserve(n * 4));
    CK(d_misc.reserve(16));
    u64* ds = d_in.as<u64>();
    u64* de = ds + n;
    CK(cudaMemcpyAsync(ds, start, n * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(de, end, n * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(d_misc.p, 0, 16, st));
    TFBS_LAUNCH(k_bed_rank, grid_for(n, BED_THREADS), BED_THREADS, 0, st)(ds, (u64)n, d_order.as<u32>());
    TFBS_LAUNCH(k_bed_merge, 1, BED_THREADS, 0, st)(ds, de, d_order.as<u32>(), (u64)n, d_out.as<u64>(), d_out.as<u64>() + n, d_misc.as<u64>(),
                                                    reinterpret_cast<u32*>(d_misc.as<u64>() + 1));
    uint64_t misc[2] = {0, 0};
    CK(cudaMemcpyAsync(misc, d_misc.p, 16, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if ((uint32_t)misc[1]) return fail(ctx, TFBS_ERR_INVALID_ARGUMENT, "a range has end < start");
    CK(cudaMemcpyAsync(out_start, d_out.p, misc[0] * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(out_end, d_out.as<u64>() + n, misc[0] * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    *n_out = misc[0];
    return TFBS_OK;
}

int tfbs_get_attribution(tfbs_ctx* ctx, tfbs_attribution* out) {
    if (!ctx || !out) return TFBS_ERR_INVALID_ARGUMENT;
    switch (ctx->att_state) {
    case tfbs_ctx::ATT_NONE: return fail(ctx, TFBS_ERR_STATE, "no block has been collected yet (tfbs_collect / tfbs_collect_grouped first)");
    case tfbs_ctx::ATT_OFF: return fail(ctx, TFBS_ERR_STATE, "option attribution was off for the last block: set it to 1 before the run");
    case tfbs_ctx::ATT_FULL_SCAN:
        return fail(ctx, TFBS_ERR_STATE, "the last block was a full scan (delta = 0 or record_matches): attribution comes from the default path only");
    default: break;
    }
    *out = ctx->att;
    return TFBS_OK;
}

int tfbs_get_sites(tfbs_ctx* ctx, tfbs_sites* out) {
    if (!ctx || !out) return TFBS_ERR_INVALID_ARGUMENT;
    switch (ctx->site_state) {
    case tfbs_ctx::ATT_NONE: return fail(ctx, TFBS_ERR_STATE, "no block has been collected yet (tfbs_collect / tfbs_collect_grouped first)");
    case tfbs_ctx::ATT_OFF: return fail(ctx, TFBS_ERR_STATE, "option sites was off for the last block: set it (and attribution) to 1 before the run");
    case tfbs_ctx::ATT_FULL_SCAN:
        return fail(ctx, TFBS_ERR_STATE, "the last block was a full scan (delta = 0, record_matches or the audit): sites come from the default path only");
    default: break;
    }
    *out = ctx->site;
    return TFBS_OK;
}

int tfbs_get_record_sites(tfbs_ctx* ctx, tfbs_record_sites* out) {
    if (!ctx || !out) return TFBS_ERR_INVALID_ARGUMENT;
    switch (ctx->rec_state) {
    case tfbs_ctx::ATT_NONE: return fail(ctx, TFBS_ERR_STATE, "no block has been collected yet (tfbs_collect / tfbs_collect_grouped first): no record sites");
    case tfbs_ctx::ATT_OFF: return fail(ctx, TFBS_ERR_STATE, "option record_sites was off for the last block: set it to 1 before the run");
    case tfbs_ctx::ATT_FULL_SCAN:
        return fail(ctx, TFBS_ERR_STATE, "the last block was a full scan (delta = 0, record_matches or the audit): record sites come from the default path only");
    default: break;
    }
    *out = ctx->rec;
    return TFBS_OK;
}

int tfbs_get_matches(tfbs_ctx* ctx, tfbs_matches* out) {
    if (!ctx || !out) return TFBS_ERR_INVALID_ARGUMENT;
    if (ctx->last < 0 || !ctx->slot[ctx->last].full_mode || !ctx->record_matches)
        return fail(ctx, TFBS_ERR_STATE, "matches were not recorded (set option record_matches before the run)");
    out->n_matches = ctx->n_matches;
    out->region = ctx->h_m_region.as<uint32_t>();
    out->pattern_index = ctx->h_m_pattern.as<uint32_t>();
    out->group = ctx->h_m_group.as<uint32_t>();
    out->start = ctx->h_m_start.as<int64_t>();
    out->hap_group = ctx->h_hap_group.as<uint32_t>();
    out->n_samples = ctx->slot[ctx->last].in->S;
    out->truncated = ctx->matches_truncated ? 1 : 0;
    return TFBS_OK;
}

// Ties = windows reported with min_score - 1 but not with min_score, i.e. score == min_score (pattern.rs:151 is strict).
int tfbs_audit_block(tfbs_ctx* ctx, tfbs_audit* out) {
    if (!ctx || !out) return TFBS_ERR_INVALID_ARGUMENT;
    memset(out, 0, sizeof *out);
    if (!ctx->last_block || !ctx->last_block->valid) return fail(ctx, TFBS_ERR_STATE, "tfbs_audit_block needs a block (tfbs_submit_block / tfbs_upload_block first)");
    if (ctx->orig_patterns.empty()) return fail(ctx, TFBS_ERR_STATE, "tfbs_set_patterns has not been called");
    CK(cudaSetDevice(ctx->device));
    BlockDev* blk = ctx->last_block;
    int rc0 = drain(ctx);  // whatever was in flight is dropped: the audit owns the device and leaves its own run behind
    if (rc0) return rc0;
    struct Hit {
        uint32_t region, pattern, group;
        int64_t start;
        bool operator<(const Hit& o) const {
            if (region != o.region) return region < o.region;
            if (pattern != o.pattern) return pattern < o.pattern;
            if (group != o.group) return group < o.group;
            return start < o.start;
        }
        bool operator==(const Hit& o) const { return region == o.region && pattern == o.pattern && group == o.group && start == o.start; }
    };
    auto take_hits = [&](std::vector<Hit>* v) {
        v->resize(ctx->n_matches);
        for (uint64_t i = 0; i < ctx->n_matches; ++i)
            (*v)[i] = Hit{ctx->h_m_region.as<uint32_t>()[i], ctx->h_m_pattern.as<uint32_t>()[i], ctx->h_m_group.as<uint32_t>()[i],
                          ctx->h_m_start.as<int64_t>()[i]};
        std::sort(v->begin(), v->end());
    };
    const int keep_record = ctx->record_matches;
    ctx->record_matches = 1;  // forces the full scan of every distinct haplotype
    ctx->audit = 1;
    std::vector<tfbs_pattern> lowered = ctx->orig_patterns;
    for (tfbs_pattern& p : lowered)
        if (p.min_score > INT32_MIN) p.min_score -= 1;  // score > INT32_MIN - 1 cannot be expressed; such a pattern has no tie list
    std::vector<Hit> with_ties, hits;
    bool overflow = false;
    const uint64_t keep_max = ctx->max_matches;
    auto run_once = [&]() -> int {
        ctx->in_flight = 0;
        ctx->head = 0;
        return start_block(ctx, blk, nullptr);
    };
    // a run that overflows the match buffer says how many hits there were: run it once more with a buffer of that size
    auto run_recorded = [&]() -> int {
        int r = run_once();
        if (r == TFBS_OK && ctx->matches_truncated && ctx->n_matches_found < (1ull << 31)) {
            ctx->max_matches = ctx->n_matches_found + ctx->n_matches_found / 8 + 1024;
            r = run_once();
        }
        return r;
    };
    int rc = install_patterns(ctx, lowered.data(), (uint32_t)lowered.size());
    if (rc == TFBS_OK) rc = run_recorded();
    if (rc == TFBS_OK) {
        take_hits(&with_ties);
        overflow = ctx->matches_truncated;
    }
    // always put the caller's thresholds back, and leave the context with a normal run of the block (tfbs_collect works)
    int rc2 = install_patterns(ctx, ctx->orig_patterns.data(), (uint32_t)ctx->orig_patterns.size());
    if (rc2 == TFBS_OK && rc == TFBS_OK) rc2 = run_recorded();
    ctx->record_matches = keep_record;
    ctx->max_matches = keep_max;
    ctx->audit = 0;
    if (rc != TFBS_OK || rc2 != TFBS_OK) {
        ctx->in_flight = 0;
        return rc != TFBS_OK ? rc : rc2;
    }
    ctx->last = 0;  // tfbs_get_matches right after the audit sees this run
    take_hits(&hits);
    overflow = overflow || ctx->matches_truncated;
    ctx->tie_region.clear();
    ctx->tie_pattern.clear();
    ctx->tie_group.clear();
    ctx->tie_start.clear();
    size_t j = 0;
    for (const Hit& h : with_ties) {  // sorted set difference
        while (j < hits.size() && hits[j] < h) ++j;
        if (j < hits.size() && hits[j] == h) continue;
        ctx->tie_region.push_back(h.region);
        ctx->tie_pattern.push_back(h.pattern);
        ctx->tie_group.push_back(h.group);
        ctx->tie_start.push_back(h.start);
    }
    out->n_ties = ctx->tie_region.size();
    out->tie_region = ctx->tie_region.data();
    out->tie_pattern_index = ctx->tie_pattern.data();
    out->tie_group = ctx->tie_group.data();
    out->tie_start = ctx->tie_start.data();
    out->hap_group = ctx->h_hap_group.as<uint32_t>();
    out->hap_flags = ctx->h_hap_flags.as<uint8_t>();
    out->n_regions = blk->R;
    out->n_samples = blk->S;
    out->truncated = overflow ? 1 : 0;
    return TFBS_OK;
}

int tfbs_get_stats(const tfbs_ctx* ctx, tfbs_stats* out) {
    if (!ctx || !out) return TFBS_ERR_INVALID_ARGUMENT;
    if (ctx->last < 0) memset(out, 0, sizeof *out);
    else *out = ctx->slot[ctx->last].stats;
    return TFBS_OK;
}

int tfbs_fanout_info(const tfbs_ctx* ctx, uint32_t* smem_groups, uint32_t* groups_cap, uint32_t* ctas, uint32_t* in_device_memory) {
    if (!ctx || !smem_groups || !groups_cap || !ctas || !in_device_memory) return TFBS_ERR_INVALID_ARGUMENT;
    *smem_groups = fan_smem_groups(ctx->prop);
    const Slot* s = ctx->last < 0 ? nullptr : &ctx->slot[ctx->last];
    const bool ran = s && !s->full_mode;
    *groups_cap = ran ? s->fan_groups_cap : 0;
    *ctas = ran ? s->fan_ctas : 0;
    *in_device_memory = ran ? s->fan_in_device_memory : 0;
    return TFBS_OK;
}

int tfbs_host_register(void* ptr, size_t bytes) {
    if (!ptr || !bytes) return TFBS_OK;
    return cudaHostRegister(ptr, bytes, cudaHostRegisterDefault) == cudaSuccess ? TFBS_OK : TFBS_ERR_CUDA;
}
int tfbs_host_unregister(void* ptr) {
    if (!ptr) return TFBS_OK;
    return cudaHostUnregister(ptr) == cudaSuccess ? TFBS_OK : TFBS_ERR_CUDA;
}

void* tfbs_stream(const tfbs_ctx* ctx) { return ctx ? (void*)ctx->lane[0].stream : nullptr; }

}  // extern "C"
