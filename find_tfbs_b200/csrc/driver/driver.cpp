// driver.cpp -- find-tfbs-b200: the reference's command line on top of libtfbs_b200.so.
//
// Host side of the hot path, mirroring the reference (Helkafen/find-tfbs) so that a user can switch binaries:
//   options            src/main.rs:169-227   (long options are the API; the colliding short flags -n / -t are not offered)
//   PWM + thresholds   src/pattern.rs:13-117
//   BED + merge        src/bed.rs:9-60, src/range.rs:18-87
//   samples            src/main.rs:293-313
//   per region glue    src/main.rs:395-436   (halo :404-407, FASTA window :156-161, select_inner_peaks :62-72,
//                                              BCF fetch + GT rule src/haplotype.rs:13-62,78-79)
//   rows               src/main.rs:415-429, counts_as_genotypes :439-498 (second half: classes, dosage, COUNTS, freqs, maf)
//   writer             src/main.rs:264-290   (BGZF .part file, rename; --tabix runs tabix on it)
// Everything between "window + records in memory" and "(left, right) count vectors" runs on the GPU through the C ABI
// (include/tfbs.h).  There is no CPU implementation of that part in this program.
//
// Third-party formats the reference reads through crates (rust-htslib 0.26.1, bio 0.28.2, bgzip 0.0.3) are decoded here
// directly: BGZF (gzip members), BCF2.2, .fai-indexed FASTA, BED.
#include "common.hpp"
#include "options.hpp"
#include "pwm.hpp"
#include "bed.hpp"
#include "bgzf.hpp"
#include "bcf.hpp"
#include "fasta.hpp"
#include "block.hpp"
#include "rows.hpp"

#ifdef TFBS_DRIVER_TEST_SHIM
#include "test_shim.hpp"
#endif

#ifndef TFBS_DRIVER_NO_MAIN
namespace {
#define TF(call)                                                         \
    do {                                                                 \
        int rc_ = (call);                                                \
        if (rc_ != TFBS_OK) die(tfbs_last_error(ctx));                   \
    } while (0)

}  // namespace

int main(int argc, char** argv) {
    Options o = parse_args(argc, argv);
    if (!o.write_thresholds.empty()) {  // threshold tooling: exact score distribution of every (wanted) PWM -> <DIR>/<name>.thr
        size_t n = 0;
        for (const auto& def : read_pwm_definitions(o.pwm_file)) {
            if (!o.pwm_names.empty() && std::find(o.pwm_names.begin(), o.pwm_names.end(), def.first) == o.pwm_names.end()) continue;
            if (def.second.empty()) continue;
            write_threshold_file(o.write_thresholds + "/" + def.first + ".thr", def.second, o.pvalues);
            ++n;
        }
        printf("Wrote %zu threshold files to %s\n", n, o.write_thresholds.c_str());
        return 0;
    }
    if (o.tabix && system("command -v tabix > /dev/null 2>&1") != 0) die("tabix cannot in found in PATH");  // main.rs:220-223
    auto t_start = std::chrono::steady_clock::now();
    auto since = [&] { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count(); };

    std::vector<Pwm> pwms = parse_pwm_files(o);
    if (pwms.empty()) die("assertion failed: pwm_list.len() > 0");  // main.rs:238
    std::map<uint16_t, std::string> pwm_name;
    uint32_t largest = 0;
    for (const Pwm& p : pwms) {
        printf("PWM %s %d %s %zu\n", p.name.c_str(), p.min_score, p.direction == TFBS_DIR_P ? "P" : "N", p.w.size() / 4);
        pwm_name[p.pattern_id] = p.name;
        largest = std::max<uint32_t>(largest, (uint32_t)(p.w.size() / 4));
    }

    // load_peak_files (bed.rs:25-60)
    std::vector<std::vector<Range>> peak_map;
    std::vector<std::string> bed_names;
    std::vector<Range> all;
    for (const std::string& b : o.beds) {
        std::vector<Range> peaks = load_bed(b, o.chromosome), kept;
        uint64_t cover = 0;
        for (const Range& p : peaks) cover += p.end - p.start;
        printf("Loaded %s:\t %zu peaks covering %llu bp\n", b.c_str(), peaks.size(), (unsigned long long)cover);
        for (const Range& p : peaks)
            if (p.start >= o.after_position) kept.push_back(p);
        all.insert(all.end(), kept.begin(), kept.end());
        peak_map.push_back(kept);
        bed_names.push_back(basename_of(b));
    }

    // one context per device; chunks of merged regions are dealt round-robin (regions are independent, main.rs:395-429)
    std::vector<tfbs_pattern> cpat(pwms.size());
    for (size_t i = 0; i < pwms.size(); ++i) {
        cpat[i].weights = pwms[i].w.data();
        cpat[i].len = (uint32_t)(pwms[i].w.size() / 4);
        cpat[i].min_score = pwms[i].min_score;
        cpat[i].pattern_id = pwms[i].pattern_id;
        cpat[i].direction = pwms[i].direction;
        cpat[i].kind = TFBS_PATTERN_PWM;
    }
    // the CUDA contexts are created (and the pattern tables compiled and uploaded) while the BCF is read
    std::atomic<uint64_t> us_create{0};
    auto now_us = [] { return (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    if (o.devices.empty()) o.devices.push_back(0);
    std::vector<tfbs_ctx*> ctxs(o.devices.size(), nullptr);
    std::vector<std::thread> pre;
    for (size_t k = 0; k < o.devices.size(); ++k)
        pre.emplace_back([&, k] {
            const uint64_t tc = now_us();
            tfbs_ctx* ctx = nullptr;
            if (tfbs_create(o.devices[k], &ctx) != TFBS_OK) die(std::string(tfbs_last_error(nullptr)));
            TF(tfbs_set_patterns(ctx, cpat.data(), (uint32_t)cpat.size()));
            TF(tfbs_set_option(ctx, "rows_width", 0));
            if (!o.attribution_file.empty()) TF(tfbs_set_option(ctx, "attribution", 1));
            ctxs[k] = ctx;
            us_create += now_us() - tc;
        });
    const double t_before_bcf = since();
    Cohort co = load_bcf(o);
    const double t_after_bcf = since();
    for (auto& t : pre) t.join();
    // the merged regions (bed.rs:37-45): on the first device; ranges with end < start only fold in file order, on the host
    std::vector<Range> merged;
    {
        std::vector<uint64_t> bs(all.size()), be(all.size()), ms(all.size()), me(all.size());
        for (size_t i = 0; i < all.size(); ++i) { bs[i] = all[i].start; be[i] = all[i].end; }
        uint64_t nm = 0;
        const int rc = ctxs[0] ? tfbs_merge_regions(ctxs[0], bs.data(), be.data(), all.size(), ms.data(), me.data(), &nm) : TFBS_ERR_INVALID_ARGUMENT;
        if (rc == TFBS_OK) {
            for (uint64_t i = 0; i < nm; ++i) merged.push_back(Range{ms[i], me[i]});
        } else if (rc == TFBS_ERR_INVALID_ARGUMENT) {
            merged = merge_ranges(all);
        } else {
            die(std::string(tfbs_last_error(ctxs[0])));
        }
    }
    printf("Merged all region files: %zu merged regions\n", merged.size());
    const uint32_t S = (uint32_t)co.samples.size();

    // main.rs:402 chromosome.replace("chr", ""): one left-to-right pass over non-overlapping matches
    std::string chr;
    for (size_t p = 0; p < o.chromosome.size();) {
        if (o.chromosome.compare(p, 3, "chr") == 0) p += 3;
        else chr += o.chromosome[p++];
    }

    const std::string part = o.output + ".part";
    BgzfWriter* gz = o.plain_text ? nullptr : new BgzfWriter(part, o.threads, o.compression_level);
    std::ofstream plain;
    if (o.plain_text) { plain.open(part, std::ios::binary); if (!plain) die("Could not create output file"); }
    auto emit = [&](const std::string& s) { if (gz) gz->write(s); else plain << s; };
    {
        std::string hdr = "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT";  // main.rs:320-324
        for (auto& s : co.samples) hdr += "\t" + s;
        emit(hdr + "\n");
    }

    // Regions per block: the reference hands out chunks of 50 (main.rs:375-381); a block here should keep a GPU busy for milliseconds
    // (thousands of regions for a small cohort) yet leave several blocks per run, so that row text, compression and the GPU overlap
    // (a region of a 2,504-sample cohort already gives ~75 rows of 25 KB).
    if (o.chunk == 0) o.chunk = (uint32_t)std::min<uint64_t>(2000, std::max<uint64_t>(50, 2000000ull / std::max<uint32_t>(1, S)));
    const size_t n_chunks = (merged.size() + o.chunk - 1) / o.chunk;
    // The writer (main.rs:264-290 has a writer thread fed through a channel): chunks finish in any order on the devices and are
    // written in chunk order as soon as every earlier chunk is there; a finished chunk's text is freed once written, so the
    // memory in flight is a few chunks, not the chromosome.  POS is the reference's running counter (main.rs:329,424-425).
    struct ChunkText { std::vector<std::string> rows; std::string attribution; };
    std::mutex out_mu;
    std::condition_variable out_cv;
    std::map<size_t, ChunkText> done_chunks;
    std::vector<std::string> audit_text(o.audit_file.empty() ? 0 : n_chunks);
    // --attribution: per written row (after --min_maf), in the VCF's order, the configurations -- records of one cluster of nearby
    // records that haplotypes carry together -- whose count difference to the reference haplotype is not 0.  A haplotype counts
    // REF_COUNT plus the DIFF of every line whose configuration it carries; HAPLOTYPES = how many selected haplotypes carry it.
    // TRUNCATES = 1: the configuration runs into patch_haplotype's truncation exit (haplotype.rs:144-149), DIFF includes the hits lost
    // behind it.  The writer thread appends a chunk's lines with its rows, so they are held for a few chunks at a time.
    std::ofstream attribution_out;
    if (!o.attribution_file.empty()) {
        attribution_out.open(o.attribution_file, std::ios::binary);
        if (!attribution_out) die("Could not create attribution file");
        attribution_out << "#ID\tREF_COUNT\tRECORDS\tDIFF\tHAPLOTYPES\tTRUNCATES\n";
    }
    size_t next_to_write = 0;
    uint64_t fake_position = 1;
    double secs_write = 0;
    // the writer thread: takes the chunks in order, numbers the rows and feeds the BGZF writer while the workers go on
    std::thread writer([&] {
        for (;;) {
            ChunkText t;
            {
                std::unique_lock<std::mutex> lk(out_mu);
                out_cv.wait(lk, [&] { return next_to_write == n_chunks || done_chunks.count(next_to_write); });
                if (next_to_write == n_chunks) return;
                auto it = done_chunks.find(next_to_write);
                t = std::move(it->second);
                done_chunks.erase(it);
            }
            auto tw = std::chrono::steady_clock::now();
            // CHROM, POS, then the row as the worker formatted it.  The rows of the chunk are cut into one range per host thread;
            // every range is assembled and compressed into BGZF blocks of its own (the blocks of a BGZF file are independent gzip
            // members), the writer only appends the finished blocks in order.
            const size_t n = t.rows.size();
            const uint64_t first = fake_position;
            fake_position += n;
            const size_t nt = std::max<size_t>(1, std::min<size_t>(o.threads, n / 64 + 1));
            std::vector<std::string> piece(nt);
            auto assemble = [&](size_t k) {
                const size_t a = n * k / nt, b = n * (k + 1) / nt;
                size_t bytes = 0;
                for (size_t i = a; i < b; ++i) bytes += t.rows[i].size() + chr.size() + 24;
                std::string text;
                text.reserve(bytes);
                for (size_t i = a; i < b; ++i) {
                    text += chr;
                    text += '\t';
                    text += std::to_string(first + i);
                    text += t.rows[i];
                    std::string().swap(t.rows[i]);  // the row's memory goes back as soon as it has been copied
                }
                piece[k] = gz ? BgzfWriter::compress_blocks(text.data(), text.size(), gz->level()) : std::move(text);
            };
            if (nt == 1) assemble(0);
            else {
                std::vector<std::thread> th;
                for (size_t k = 0; k < nt; ++k) th.emplace_back(assemble, k);
                for (auto& x : th) x.join();
            }
            for (const std::string& pc : piece) {
                if (gz) gz->write_blocks(pc);
                else plain << pc;
            }
            if (attribution_out.is_open()) attribution_out << t.attribution;
            secs_write += std::chrono::duration<double>(std::chrono::steady_clock::now() - tw).count();
            {
                std::lock_guard<std::mutex> lk(out_mu);
                ++next_to_write;
            }
            out_cv.notify_all();
        }
    });
    // a worker hands a finished chunk over; it waits while the writer is more than a few chunks behind (bounded memory)
    auto chunk_finished = [&](size_t c, ChunkText&& t) {
        std::unique_lock<std::mutex> lk(out_mu);
        out_cv.wait(lk, [&] { return c < next_to_write + 8 + 2 * o.devices.size(); });
        done_chunks.emplace(c, std::move(t));
        out_cv.notify_all();
    };

    std::atomic<size_t> next{0};
    std::atomic<uint64_t> total_cells{0}, total_hits{0};
    std::atomic<uint64_t> us_wait{0}, us_gpu{0}, us_sort{0}, us_format{0};
    auto worker = [&](size_t slot) {
        tfbs_ctx* ctx = ctxs[slot];
        // a builder thread prepares the next blocks (FASTA windows, inner regions, records) while the GPU works on the current one;
        // private readers per worker, like main.rs:345-346
        struct Ready { size_t c = 0; std::unique_ptr<BlockData> bd; };
        std::mutex mu;
        std::condition_variable cv;
        std::deque<Ready> ready;
        bool finished = false;
        std::thread builder([&] {
            Fasta fa(o.reference, o.chromosome);
            for (;;) {
                size_t c = next.fetch_add(1);
                if (c >= n_chunks) break;
                std::unique_ptr<BlockData> bd(new BlockData());
                build_block(merged, c * o.chunk, std::min(merged.size(), (c + 1) * (size_t)o.chunk), peak_map, co, fa, largest, bd.get());
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return ready.size() < 3; });
                ready.push_back(Ready{c, std::move(bd)});
                cv.notify_all();
            }
            std::lock_guard<std::mutex> lk(mu);
            finished = true;
            cv.notify_all();
        });
        auto take_ready = [&](Ready* item, bool wait) -> bool {
            uint64_t tw = now_us();
            std::unique_lock<std::mutex> lk(mu);
            if (wait) cv.wait(lk, [&] { return !ready.empty() || finished; });
            if (ready.empty()) return false;
            *item = std::move(ready.front());
            ready.pop_front();
            cv.notify_all();
            us_wait += now_us() - tw;
            return true;
        };
        // rows of one block -> text, in the canonical order inside a region: (bed file, inner range, pattern_id); the reference's
        // order is HashMap::drain().  `counts(i, l, r)` fills the (left, right) vectors of row i; `attribution(i, id, text)`, when
        // given, appends the --attribution lines of a written row i with VCF ID `id`.
        using AttributionLines = std::function<void(uint64_t, const std::string&, std::string&)>;
        auto rows_to_text = [&](size_t c, const BlockData& bd, uint64_t n_rows, const uint32_t* region, const uint32_t* inner, const uint16_t* pid,
                                const uint32_t* vmin, const uint32_t* vmax, const std::function<void(uint64_t, uint32_t*, uint32_t*)>& counts,
                                const AttributionLines& attribution = nullptr) {
            uint64_t ts = now_us();
            std::vector<uint64_t> order(n_rows);
            for (uint64_t i = 0; i < n_rows; ++i) order[i] = i;
            std::stable_sort(order.begin(), order.end(), [&](uint64_t a, uint64_t b) {
                if (region[a] != region[b]) return region[a] < region[b];
                const tfbs_inner_region& ia = bd.inner[inner[a]];
                const tfbs_inner_region& ib = bd.inner[inner[b]];
                if (ia.bed_index != ib.bed_index) return ia.bed_index < ib.bed_index;
                if (ia.start != ib.start) return ia.start < ib.start;
                if (ia.end != ib.end) return ia.end < ib.end;
                return pid[a] < pid[b];
            });
            us_sort += now_us() - ts;
            uint64_t tf = now_us();
            // row text on --threads host threads (the reference formats inside its worker threads, main.rs:415-425)
            std::vector<std::string> text(order.size()), att(attribution ? order.size() : 0);
            auto format_range = [&](size_t a, size_t b) {
                std::vector<uint32_t> l(S), r(S);
                for (size_t k = a; k < b; ++k) {
                    const uint64_t i = order[k];
                    counts(i, l.data(), r.data());
                    RowText t = finalise_row(l.data(), r.data(), S, vmin[i], vmax[i], o.min_maf);
                    if (!t.keep) continue;
                    const tfbs_inner_region& ir = bd.inner[inner[i]];
                    const std::string id = bed_names[ir.bed_index] + "," + pwm_name.at(pid[i]) + "," + std::to_string(ir.start) + "-" + std::to_string(ir.end);
                    // POS is filled in by the writer (a running counter, main.rs:329,424-425)
                    text[k] = "\t" + id + "\t.\t.\t.\tPASS\t" + t.info + "\tGT:DS" + t.genotypes + "\n";
                    if (attribution) attribution(i, id, att[k]);
                }
            };
            const size_t nt = std::max<size_t>(1, std::min<size_t>(o.threads, order.size() / 64 + 1));
            if (nt == 1) format_range(0, order.size());
            else {
                std::vector<std::thread> ft;
                for (size_t t = 0; t < nt; ++t) ft.emplace_back(format_range, order.size() * t / nt, order.size() * (t + 1) / nt);
                for (auto& t : ft) t.join();
            }
            ChunkText ct;
            for (std::string& row : text)
                if (!row.empty()) ct.rows.push_back(std::move(row));
            for (const std::string& a : att) ct.attribution += a;
            us_format += now_us() - tf;
            chunk_finished(c, std::move(ct));
        };
        auto note_stats = [&](size_t c) {
            tfbs_stats st;
            tfbs_get_stats(ctx, &st);
            total_cells += st.nominal_cells;
            total_hits += st.n_hits;
            if (o.verbose)
                printf("\nChunk %zu/%zu\t%llu haplotypes\t%llu hits\n", c + 1, n_chunks, (unsigned long long)st.n_groups, (unsigned long long)st.n_hits);
        };
        if (o.audit_file.empty()) {
            // The rows of a collected block are copied out of the library's buffers (they are reused by the next collect) and handed
            // to a formatter thread: sorting and row text of block c run while this thread submits and collects the next blocks.
            struct OwnedRows {
                std::vector<uint32_t> region, inner, vmin, vmax, base, packed, n_groups;
                std::vector<uint16_t> pid;
                std::vector<uint8_t> bits, hap_group;
                std::vector<uint64_t> offset;
                tfbs_grouped_rows g{};
                explicit OwnedRows(const tfbs_grouped_rows& s) {
                    const uint64_t n = s.n_rows, RH = (uint64_t)s.n_regions * 2 * s.n_samples;
                    region.assign(s.region, s.region + n); inner.assign(s.inner, s.inner + n); pid.assign(s.pattern_id, s.pattern_id + n);
                    vmin.assign(s.vmin, s.vmin + n); vmax.assign(s.vmax, s.vmax + n); base.assign(s.base, s.base + n);
                    bits.assign(s.bits, s.bits + n); offset.assign(s.offset, s.offset + n);
                    packed.assign(s.packed, s.packed + s.packed_words);
                    n_groups.assign(s.n_groups, s.n_groups + s.n_regions);
                    hap_group.assign((const uint8_t*)s.hap_group, (const uint8_t*)s.hap_group + RH * s.hap_group_bytes);
                    g = s;
                    g.region = region.data(); g.inner = inner.data(); g.pattern_id = pid.data(); g.vmin = vmin.data(); g.vmax = vmax.data();
                    g.base = base.data(); g.bits = bits.data(); g.offset = offset.data(); g.packed = packed.data();
                    g.n_groups = n_groups.data(); g.hap_group = hap_group.data();
                }
            };
            // --attribution: the block's attribution, copied like the rows, and per configuration the haplotypes whose group lists it
            struct OwnedAttribution {
                std::vector<uint32_t> ref_count, term_cfg, cfg_rec;
                std::vector<int32_t> term_diff;
                std::vector<uint64_t> term_off, cfg_rec_off, haplotypes;
                std::vector<uint8_t> cfg_flags;
                OwnedAttribution(const tfbs_attribution& a, const tfbs_grouped_rows& g) {
                    const uint64_t n = a.n_rows, nt = a.term_off[n], nc = a.n_cfgs;
                    ref_count.assign(a.ref_count, a.ref_count + n);
                    term_off.assign(a.term_off, a.term_off + n + 1);
                    term_cfg.assign(a.term_cfg, a.term_cfg + nt);
                    term_diff.assign(a.term_diff, a.term_diff + nt);
                    cfg_flags.assign(a.cfg_flags, a.cfg_flags + nc);
                    cfg_rec_off.assign(a.cfg_rec_off, a.cfg_rec_off + nc + 1);
                    cfg_rec.assign(a.cfg_rec, a.cfg_rec + cfg_rec_off[nc]);
                    // haplotypes per group (block-wide group index), then per configuration over the groups that list it
                    const uint64_t H = 2ull * g.n_samples;
                    std::vector<uint64_t> members(a.n_groups_total, 0);
                    uint64_t gb = 0;
                    for (uint32_t r = 0; r < g.n_regions && a.n_groups_total; ++r) {
                        for (uint64_t h = 0; h < H; ++h) {
                            const uint64_t x = r * H + h;
                            ++members[gb + (g.hap_group_bytes == 2 ? ((const uint16_t*)g.hap_group)[x] : ((const uint32_t*)g.hap_group)[x])];
                        }
                        gb += g.n_groups[r];
                    }
                    haplotypes.assign(nc, 0);
                    for (uint64_t G = 0; G < a.n_groups_total; ++G)
                        for (uint64_t k = a.group_cfg_off[G]; k < a.group_cfg_off[G + 1]; ++k) haplotypes[a.group_cfg[k]] += members[G];
                }
            };
            struct Collected { size_t c; std::unique_ptr<BlockData> bd; std::unique_ptr<OwnedRows> rows; std::unique_ptr<OwnedAttribution> att; };
            std::mutex fmu;
            std::condition_variable fcv;
            std::deque<Collected> to_format;
            bool collected_all = false;
            std::thread formatter([&] {
                for (;;) {
                    Collected it;
                    {
                        std::unique_lock<std::mutex> lk(fmu);
                        fcv.wait(lk, [&] { return !to_format.empty() || collected_all; });
                        if (to_format.empty()) return;
                        it = std::move(to_format.front());
                        to_format.pop_front();
                        fcv.notify_all();
                    }
                    const tfbs_grouped_rows& g = it.rows->g;
                    const OwnedAttribution* at = it.att.get();
                    const BlockData& bd = *it.bd;
                    // ID, REF_COUNT, RECORDS (POS:REF:ALT, 1-based POS), DIFF, HAPLOTYPES, TRUNCATES: one line per term of the row
                    auto lines = [&](uint64_t i, const std::string& id, std::string& out) {
                        for (uint64_t t = at->term_off[i]; t < at->term_off[i + 1]; ++t) {
                            const uint32_t cfg = at->term_cfg[t];
                            std::string recs;
                            for (uint64_t k = at->cfg_rec_off[cfg]; k < at->cfg_rec_off[cfg + 1]; ++k) {
                                const tfbs_variant& v = bd.variants[at->cfg_rec[k]];
                                if (!recs.empty()) recs += ';';
                                recs += std::to_string(v.pos + 1) + ":" + std::string((const char*)bd.alleles.data() + v.ref_off, v.ref_len) + ":" +
                                        std::string((const char*)bd.alleles.data() + v.alt_off, v.alt_len);
                            }
                            out += id + "\t" + std::to_string(at->ref_count[i]) + "\t" + recs + "\t" + std::to_string(at->term_diff[t]) + "\t" +
                                   std::to_string(at->haplotypes[cfg]) + "\t" + ((at->cfg_flags[cfg] & TFBS_CFG_TRUNCATES) ? "1" : "0") + "\n";
                        }
                    };
                    rows_to_text(it.c, bd, g.n_rows, g.region, g.inner, g.pattern_id, g.vmin, g.vmax,
                                 [&](uint64_t i, uint32_t* l, uint32_t* r) { tfbs_expand_rows(&g, i, 1, l, r); }, at ? AttributionLines(lines) : nullptr);
                }
            });
            // two blocks in flight per device: the copies and the host work of one overlap the kernels of the other
            std::deque<Ready> flying;
            for (;;) {
                while (flying.size() < 2) {
                    Ready item;
                    if (!take_ready(&item, flying.empty())) break;
                    uint64_t tg = now_us();
                    tfbs_block blk = item.bd->view(co);
                    TF(tfbs_submit_block(ctx, &blk));
                    us_gpu += now_us() - tg;
                    flying.push_back(std::move(item));
                }
                if (flying.empty()) break;
                Ready item = std::move(flying.front());
                flying.pop_front();
                uint64_t tg = now_us();
                tfbs_grouped_rows g;
                TF(tfbs_collect_grouped(ctx, &g));
                us_gpu += now_us() - tg;
                note_stats(item.c);
                std::unique_ptr<OwnedRows> own(new OwnedRows(g));
                std::unique_ptr<OwnedAttribution> att;
                if (!o.attribution_file.empty()) {
                    tfbs_attribution a;
                    TF(tfbs_get_attribution(ctx, &a));
                    att.reset(new OwnedAttribution(a, g));
                }
                std::unique_lock<std::mutex> lk(fmu);
                fcv.wait(lk, [&] { return to_format.size() < 2; });  // bounded: at most two collected blocks wait for their text
                to_format.push_back(Collected{item.c, std::move(item.bd), std::move(own), std::move(att)});
                fcv.notify_all();
            }
            {
                std::lock_guard<std::mutex> lk(fmu);
                collected_all = true;
            }
            fcv.notify_all();
            formatter.join();
        } else {
            for (;;) {
                Ready item;
                if (!take_ready(&item, true)) break;
                const size_t c = item.c, m0 = c * o.chunk;
                BlockData& bd = *item.bd;
                uint64_t tg = now_us();
                tfbs_block blk = bd.view(co);
                // the audit scores the block twice (thresholds lowered by one, then as given) and leaves the rows of the normal run
                TF(tfbs_upload_block(ctx, &blk));
                tfbs_audit au;
                TF(tfbs_audit_block(ctx, &au));
                if (au.truncated) die("--audit: the match buffer overflowed; use a smaller --chunk");
                std::string& out = audit_text[c];
                const uint32_t H = 2 * au.n_samples;
                auto region_name = [&](uint32_t r) { return std::to_string(merged[m0 + r].start) + "-" + std::to_string(merged[m0 + r].end); };
                for (uint64_t i = 0; i < au.n_ties; ++i) {
                    const uint32_t r = au.tie_region[i], g = au.tie_group[i];
                    uint32_t first = UINT32_MAX, members = 0;  // the group's first haplotype names it
                    for (uint32_t h = 0; h < H; ++h)
                        if (au.hap_group[(size_t)r * H + h] == g) { if (first == UINT32_MAX) first = h; ++members; }
                    const Pwm& pw = pwms[au.tie_pattern_index[i]];
                    out += "tie\t" + chr + "\t" + region_name(r) + "\t" + pw.name + "\t" + (pw.direction == TFBS_DIR_P ? "P" : "N") + "\t" +
                           std::to_string(au.tie_start[i]) + "\t" + std::to_string(pw.min_score) + "\t" +
                           (g == 0 ? std::string("reference") : co.samples[first / 2] + (first % 2 ? ":R" : ":L")) + "\t" + std::to_string(members) + "\n";
                }
                for (uint32_t r = 0; r < au.n_regions; ++r)
                    for (uint32_t h = 0; h < H; ++h) {
                        const uint8_t fl = au.hap_flags[(size_t)r * H + h];
                        if (fl & TFBS_HAP_TRUNCATED)
                            out += "truncated\t" + chr + "\t" + region_name(r) + "\t" + co.samples[h / 2] + (h % 2 ? ":R" : ":L") + "\n";
                        if (fl & TFBS_HAP_OVERWRITTEN)
                            out += "overwritten\t" + chr + "\t" + region_name(r) + "\t" + co.samples[h / 2] + (h % 2 ? ":R" : ":L") + "\n";
                    }
                tfbs_rows rows;
                TF(tfbs_collect(ctx, &rows));
                us_gpu += now_us() - tg;
                note_stats(c);
                rows_to_text(c, bd, rows.n_rows, rows.region, rows.inner, rows.pattern_id, rows.vmin, rows.vmax, [&](uint64_t i, uint32_t* l, uint32_t* r) {
                    for (uint32_t s = 0; s < S; ++s) {  // counts arrive in the narrowest type that holds them (tfbs_rows.count_bytes)
                        l[s] = rows.count_bytes == 1 ? ((const uint8_t*)rows.left)[i * S + s] : rows.count_bytes == 2 ? ((const uint16_t*)rows.left)[i * S + s] : rows.left[i * S + s];
                        r[s] = rows.count_bytes == 1 ? ((const uint8_t*)rows.right)[i * S + s] : rows.count_bytes == 2 ? ((const uint16_t*)rows.right)[i * S + s] : rows.right[i * S + s];
                    }
                });
            }
        }
        builder.join();
        tfbs_destroy(ctx);
    };
    if (o.devices.size() <= 1) worker(0);
    else {
        std::vector<std::thread> th;
        for (size_t k = 0; k < o.devices.size(); ++k) th.emplace_back(worker, k);
        for (auto& t : th) t.join();
    }
    const double t_after_gpu = since();
    writer.join();
    if (next_to_write != n_chunks) die("internal error: " + std::to_string(n_chunks - next_to_write) + " chunks were not written");
    if (gz) { gz->finish(); delete gz; } else plain.close();
    if (!o.audit_file.empty()) {
        // tie: a window scoring exactly min_score (not a hit, pattern.rs:151); truncated: haplotype.rs:144-149; overwritten: the
        // haplotype's entry of the sequence-keyed map was replaced (haplotype.rs:84), it is counted with the reference haplotype and
        // the reference program's choice between the colliding entries depends on HashMap order
        std::ofstream af(o.audit_file, std::ios::binary);
        if (!af) die("Could not create audit file");
        af << "#tie\tCHROM\tREGION\tPWM\tSTRAND\tSTART\tMIN_SCORE\tGROUP\tHAPLOTYPES\n#truncated|overwritten\tCHROM\tREGION\tHAPLOTYPE\n";
        for (const std::string& t : audit_text) af << t;
    }
    if (attribution_out.is_open()) {
        attribution_out.close();
        if (!attribution_out) die("Could not write attribution file");
    }
    if (rename(part.c_str(), o.output.c_str()) != 0) die("Could not rename " + part + " into " + o.output);
    if (o.tabix) {
        std::string cmd = "tabix -f -p vcf '" + o.output + "'";
        if (system(cmd.c_str()) == 0) printf("Tabixed file %s\n", o.output.c_str());
        else printf("Failed to tabix file %s\n", o.output.c_str());
    }
    double secs = since();
    printf("phases: PWM+BED %.2f s, BCF %.2f s, blocks+GPU+rows %.2f s (context %.2f, waiting for blocks %.2f, submit+collect %.2f, sort %.2f, "
           "row text %.2f; summed over devices), VCF writer thread %.2f s (overlapped), closing the file %.2f s\n", t_before_bcf, t_after_bcf - t_before_bcf, t_after_gpu - t_after_bcf,
           us_create / 1e6, us_wait / 1e6, us_gpu / 1e6, us_sort / 1e6, us_format / 1e6, secs_write, secs - t_after_gpu);
    printf("%zu merged regions, %llu rows, %llu hits, %.3e nominal cells in %.2f s\nEnd of program.\n", merged.size(),
           (unsigned long long)(fake_position - 1), (unsigned long long)total_hits.load(), (double)total_cells.load(), secs);
    return 0;
}
#endif
