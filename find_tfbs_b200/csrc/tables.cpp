// tables.cpp -- see tables.hpp.
#include "tables.hpp"

#include <algorithm>
#include <map>

namespace tfbs {

namespace {

struct FieldPlan {
    bool zero = false;       // contributions forced to 0 (always-hit or never-hit pattern)
    int64_t bias = 0;        // added to the first pair
    std::vector<int64_t> m;  // per column bias (<= 0)
};

// Decide how pattern p fits a field of `bits` bits whose top bit is the hit flag.
bool plan_field(const HostPattern& p, int bits, FieldPlan* fp) {
    const int64_t FLAG = int64_t(1) << (bits - 1);
    fp->m.assign(p.len, 0);
    int64_t M = 0, bmax = 0;
    for (uint32_t c = 0; c < p.len; ++c) {
        int64_t lo = 0, hi = 0;  // the N slot scores 0 (types.rs:110)
        for (int x = 0; x < 4; ++x) {
            lo = std::min<int64_t>(lo, p.w[4 * c + x]);
            hi = std::max<int64_t>(hi, p.w[4 * c + x]);
        }
        fp->m[c] = lo;
        M += lo;
        bmax += hi - lo;
    }
    const int64_t thr = int64_t(p.min_score) - M;  // biased score must be > thr
    fp->zero = false;
    if (thr < 0) {  // every window hits
        fp->zero = true;
        fp->bias = FLAG;
        return true;
    }
    if (thr >= bmax) {  // no window can hit
        fp->zero = true;
        fp->bias = 0;
        return true;
    }
    if (thr > FLAG - 1 || bmax - thr > FLAG) return false;
    fp->bias = FLAG - 1 - thr;
    return true;
}

struct Slot {
    int pattern = -1;
    FieldPlan plan;
};

}  // namespace

int compile_patterns(const tfbs_pattern* patterns, uint32_t n, uint32_t table_budget_bytes, int force_wide,
                     CompiledPatterns* out, std::string* err) {
    CompiledPatterns cp;
    std::map<uint16_t, uint32_t> pid_index;
    for (uint32_t i = 0; i < n; ++i) {
        const tfbs_pattern& s = patterns[i];
        HostPattern p;
        p.kind = s.kind;
        p.pattern_id = s.pattern_id;
        p.direction = s.direction;
        p.min_score = s.min_score;
        if (s.kind == TFBS_PATTERN_PWM) {
            if (s.len == 0 || s.weights == nullptr) {
                *err = "pattern " + std::to_string(i) + ": a PWM needs at least one column";
                return TFBS_ERR_INVALID_ARGUMENT;
            }
            if (s.len > (uint32_t)kMaxPatternLen) {
                *err = "pattern " + std::to_string(i) + ": length " + std::to_string(s.len) + " exceeds the supported maximum of " +
                       std::to_string(kMaxPatternLen) + " columns";
                return TFBS_ERR_INVALID_ARGUMENT;
            }
            p.len = s.len;
            p.w.assign(s.weights, s.weights + 4 * (size_t)s.len);
        } else if (s.kind == TFBS_PATTERN_OTHER) {
            p.len = 0;  // types.rs:97-99
        } else {
            *err = "pattern " + std::to_string(i) + ": unknown kind";
            return TFBS_ERR_INVALID_ARGUMENT;
        }
        pid_index[p.pattern_id] = 0;
        cp.patterns.push_back(std::move(p));
    }
    for (auto& kv : pid_index) {
        kv.second = (uint32_t)cp.pid_list.size();
        cp.pid_list.push_back(kv.first);
    }
    for (HostPattern& p : cp.patterns) {
        p.pid_index = pid_index[p.pattern_id];
        cp.pat_len.push_back(p.len);
        cp.pat_pid_index.push_back(p.pid_index);
        cp.pat_w.insert(cp.pat_w.end(), p.w.begin(), p.w.end());
        cp.pat_w.resize(cp.pat_w.size() + (4 * (size_t)kMaxPatternLen - p.w.size()), 0);
        cp.max_len = std::max(cp.max_len, p.len);
        if (p.kind == TFBS_PATTERN_PWM) {
            cp.sum_len += p.len;
            cp.sum_len_sq += (uint64_t)p.len * (p.len - 1);
        }
    }

    // PWM patterns by pid_index; a chunk is a contiguous pid range so that the forward and the
    // reverse-complement pattern of one PWM (same pattern_id, pattern.rs:73-77) are counted by one CTA.
    std::vector<std::vector<int>> by_pid(cp.pid_list.size());
    for (size_t i = 0; i < cp.patterns.size(); ++i)
        if (cp.patterns[i].kind == TFBS_PATTERN_PWM) by_pid[cp.patterns[i].pid_index].push_back((int)i);

    auto build_chunk = [&](uint32_t pid_lo, uint32_t pid_hi, int fields, bool dry, uint32_t* bytes_out) -> int {
        std::vector<int> ps;
        for (uint32_t q = pid_lo; q < pid_hi; ++q) ps.insert(ps.end(), by_pid[q].begin(), by_pid[q].end());
        std::stable_sort(ps.begin(), ps.end(), [&](int a, int b) { return cp.patterns[a].len > cp.patterns[b].len; });
        const int bits = fields == 3 ? 21 : 32;
        uint32_t n_trip = (uint32_t)((ps.size() + fields - 1) / fields);
        uint32_t words = 0;
        std::vector<uint32_t> tg(n_trip);
        for (uint32_t t = 0; t < n_trip; ++t) {
            uint32_t L = cp.patterns[ps[(size_t)t * fields]].len;  // longest of the triple (sorted)
            tg[t] = (L + 1) / 2;
            words += tg[t] * kPairEntries;
        }
        if (bytes_out) *bytes_out = words * 8;
        if (dry) return TFBS_OK;

        ChunkDesc cd{};
        cd.tbl_off = (uint32_t)cp.table.size();
        cd.tbl_words = words;
        cd.trip_off = (uint32_t)(cp.trip_pat.size() / 3);
        cd.n_triples = n_trip;
        cd.run_off = (uint32_t)cp.runs.size();
        cd.pid_lo = pid_lo;
        cd.n_pid = pid_hi - pid_lo;
        cd.fields = (uint32_t)fields;
        for (uint32_t t = 0; t < n_trip; ++t) {
            Slot slot[3];
            for (int f = 0; f < fields; ++f) {
                size_t k = (size_t)t * fields + f;
                if (k >= ps.size()) continue;
                slot[f].pattern = ps[k];
                if (!plan_field(cp.patterns[ps[k]], bits, &slot[f].plan)) {
                    *err = "pattern " + std::to_string(ps[k]) + ": score range does not fit a " + std::to_string(bits) + "-bit field";
                    return TFBS_ERR_SCORE_RANGE;
                }
            }
            for (int f = 0; f < 3; ++f) cp.trip_pat.push_back(slot[f].pattern);
            if (cp.runs.size() == cd.run_off || cp.runs.back().groups != tg[t]) cp.runs.push_back(RunDesc{tg[t], 0});
            cp.runs.back().n_triples++;
            for (uint32_t g = 0; g < tg[t]; ++g) {
                const size_t base = cp.table.size();
                cp.table.resize(base + kPairEntries, 0);
                for (int a = 0; a < 5; ++a)
                    for (int b = 0; b < 5; ++b) {
                        uint64_t word = 0;
                        for (int f = 0; f < fields; ++f) {
                            if (slot[f].pattern < 0) continue;
                            const HostPattern& p = cp.patterns[slot[f].pattern];
                            const FieldPlan& fp = slot[f].plan;
                            int64_t v = 0;
                            if (!fp.zero) {
                                uint32_t c0 = 2 * g, c1 = 2 * g + 1;
                                if (c0 < p.len) v += (a < 4 ? p.w[4 * c0 + a] : 0) - fp.m[c0];
                                if (c1 < p.len) v += (b < 4 ? p.w[4 * c1 + b] : 0) - fp.m[c1];
                            }
                            if (g == 0) v += fp.bias;
                            word += (uint64_t)v << (bits * f);
                        }
                        cp.table[base + pair_entry(a, b)] = word;
                    }
            }
        }
        cd.n_runs = (uint32_t)cp.runs.size() - cd.run_off;
        if (cp.table.size() & 1) cp.table.push_back(0);  // chunks start 16-byte aligned (128-bit copies into shared memory)
        cp.chunks.push_back(cd);
        cp.max_chunk_bytes = std::max(cp.max_chunk_bytes, words * 8);
        return TFBS_OK;
    };

    // Does every pattern fit the 21-bit fields?  Otherwise the whole list uses two 32-bit fields.
    int fields = 3;
    if (force_wide) fields = 2;
    else
        for (const HostPattern& p : cp.patterns) {
            FieldPlan fp;
            if (p.kind == TFBS_PATTERN_PWM && !plan_field(p, 21, &fp)) fields = 2;
        }

    cp.fields = (uint32_t)fields;
    uint32_t n_pid = (uint32_t)cp.pid_list.size();
    uint32_t lo = 0;
    while (lo < n_pid) {
        uint32_t hi = lo + 1;
        uint32_t bytes = 0;
        build_chunk(lo, hi, fields, true, &bytes);
        if (bytes > table_budget_bytes) {
            *err = "the tables of pattern_id " + std::to_string(cp.pid_list[lo]) + " alone exceed the shared-memory budget";
            return TFBS_ERR_INVALID_ARGUMENT;
        }
        while (hi < n_pid) {
            uint32_t b2 = 0;
            build_chunk(lo, hi + 1, fields, true, &b2);
            if (b2 > table_budget_bytes) break;
            ++hi;
        }
        // skip pid ranges without any PWM (OtherPattern only): nothing to scan
        bool any = false;
        for (uint32_t q = lo; q < hi; ++q) any |= !by_pid[q].empty();
        if (any) {
            int rc = build_chunk(lo, hi, fields, false, nullptr);
            if (rc != TFBS_OK) return rc;
        }
        lo = hi;
    }
    *out = std::move(cp);
    return TFBS_OK;
}

}  // namespace tfbs
