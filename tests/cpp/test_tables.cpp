// CPU check of the product's host-side pattern compiler (find_tfbs_b200/csrc/tables.cpp): the packed pair tables must flag a
// window iff its exact i32 score exceeds min_score (reference src/pattern.rs:125-129,151), for every pattern length 1..32, with
// N bases (score 0, src/types.rs:110), in both field formats, with several chunks, and with always/never-hit thresholds.
// The arithmetic below is what k_scan does per lane: acc = sum_g table[triple][g][pair_entry(code[i+2g], code[i+2g+1])].
#include <cstdio>
#include <cstdlib>
#include <random>
#include <vector>

#include "../../find_tfbs_b200/csrc/tables.hpp"

using namespace tfbs;

static int check(const std::vector<tfbs_pattern>& pats, uint32_t budget, int force_wide, std::mt19937_64& rng, const char* what,
                 const std::vector<std::vector<uint8_t>>& plant = {}) {
    CompiledPatterns cp;
    std::string err;
    int rc = compile_patterns(pats.data(), (uint32_t)pats.size(), budget, force_wide, &cp, &err);
    if (rc != TFBS_OK) { printf("FAIL %s: compile error %d %s\n", what, rc, err.c_str()); return 1; }
    const int bits = cp.fields == 3 ? 21 : 32;
    std::vector<uint8_t> seq(600);
    for (auto& c : seq) c = (rng() % 23 == 0) ? 4 : (uint8_t)(rng() % 4);
    for (size_t k = 0; k < plant.size(); ++k)  // windows placed on purpose, 40 bases apart
        for (size_t c = 0; c < plant[k].size(); ++c) seq[40 + 40 * k + c] = plant[k][c];
    std::vector<int> seen(pats.size(), 0);
    long long n_hits = 0;
    for (const ChunkDesc& cd : cp.chunks) {
        size_t word = cd.tbl_off;
        uint32_t t = 0;
        for (uint32_t rn = 0; rn < cd.n_runs; ++rn) {
            const RunDesc rd = cp.runs[cd.run_off + rn];
            for (uint32_t k = 0; k < rd.n_triples; ++k, ++t) {
                for (size_t i = 0; i < seq.size(); ++i) {
                    uint64_t acc = 0;
                    for (uint32_t g = 0; g < rd.groups; ++g) {
                        int a = i + 2 * g < seq.size() ? seq[i + 2 * g] : 4, b = i + 2 * g + 1 < seq.size() ? seq[i + 2 * g + 1] : 4;
                        acc += cp.table[word + (size_t)g * kPairEntries + pair_entry(a, b)];
                    }
                    for (uint32_t f = 0; f < cp.fields; ++f) {
                        int pi = cp.trip_pat[(size_t)(cd.trip_off + t) * 3 + f];
                        bool flag = (acc >> (bits * f + bits - 1)) & 1;
                        if (pi < 0) { if (flag) { printf("FAIL %s: empty slot flagged\n", what); return 1; } continue; }
                        const tfbs_pattern& p = pats[pi];
                        if (i == 0) seen[pi]++;
                        if (i + p.len > seq.size()) continue;  // incomplete windows are filtered in the rare path
                        long long score = 0;
                        for (uint32_t c = 0; c < p.len; ++c) score += seq[i + c] < 4 ? p.weights[4 * c + seq[i + c]] : 0;
                        bool hit = score > p.min_score;
                        n_hits += hit;
                        if (hit != flag) {
                            printf("FAIL %s: pattern %d len %u window %zu score %lld min_score %d flag %d\n", what, pi, p.len, i, score, p.min_score, (int)flag);
                            return 1;
                        }
                    }
                }
                word += (size_t)rd.groups * kPairEntries;
            }
        }
        if (t != cd.n_triples) { printf("FAIL %s: run/triple bookkeeping\n", what); return 1; }
        if (cd.tbl_off % 2) { printf("FAIL %s: chunk not 16-byte aligned\n", what); return 1; }
    }
    for (size_t i = 0; i < pats.size(); ++i)
        if (pats[i].kind == TFBS_PATTERN_PWM && seen[i] != 1) { printf("FAIL %s: pattern %zu appears %d times\n", what, i, seen[i]); return 1; }
    printf("ok %s: %zu patterns, %zu chunks, fields %u, %lld hits\n", what, pats.size(), cp.chunks.size(), cp.fields, n_hits);
    return 0;
}

int main() {
    std::mt19937_64 rng(12345);
    int bad = 0;
    for (int round = 0; round < 6; ++round) {
        std::vector<std::vector<int32_t>> store;
        std::vector<tfbs_pattern> pats;
        int n = 5 + (int)(rng() % 60);
        int scale = round == 3 ? 60000 : (round == 4 ? 3 : 6000);  // 3: too wide for 21-bit fields; 4: tiny weights
        for (int k = 0; k < n; ++k) {
            uint32_t L = round == 5 ? 1 + (uint32_t)(k % 32) : 1 + (uint32_t)(rng() % 32);
            std::vector<int32_t> w(4 * L);
            long long best = 0, worst = 0;
            for (uint32_t c = 0; c < L; ++c) {
                int mx = -1000000000, mn = 1000000000;
                for (int x = 0; x < 4; ++x) {
                    int v = (int)((long long)(rng() % (2 * scale + 1)) - scale - scale / 3);
                    w[4 * c + x] = v;
                    mx = v > mx ? v : mx;
                    mn = v < mn ? v : mn;
                }
                best += mx > 0 ? mx : 0;  // N scores 0
                worst += mn < 0 ? mn : 0;
            }
            store.push_back(w);
            tfbs_pattern p{};
            p.weights = store.back().data();
            p.len = L;
            long long span = best - worst;
            int mode = (int)(rng() % 10);
            p.min_score = mode == 0 ? (int)(worst - 5) : mode == 1 ? (int)(best + 5) : mode == 2 ? (int)best - 1 : (int)(worst + span * (30 + (long long)(rng() % 60)) / 100);
            p.pattern_id = (uint16_t)(k / 2);
            p.direction = (uint8_t)(k & 1);
            p.kind = TFBS_PATTERN_PWM;
            pats.push_back(p);
        }
        tfbs_pattern other{};
        other.kind = TFBS_PATTERN_OTHER;
        other.pattern_id = 999;
        pats.push_back(other);
        for (size_t i = 0; i + 1 < pats.size(); ++i) pats[i].weights = store[i].data();
        char name[64];
        snprintf(name, sizeof name, "round %d (auto)", round);
        bad += check(pats, 96 * 1024, 0, rng, name);
        snprintf(name, sizeof name, "round %d (wide, 12 KB chunks)", round);
        bad += check(pats, 12 * 1024, 1, rng, name);
    }
    // the format decision at the field capacity: slot 0 of three length-4 patterns has bmax = 2^20 + 2^19 (21-bit set) or
    // 2^31 + 2^29 (32-bit set); the best window B (bmax) and the worst window W (score M) are placed in the sequence, and slot 1
    // scores exactly its min_score on B, so that a carry out of slot 0's field would flag it.
    {
        const int best[4] = {0, 1, 2, 3}, worst[4] = {3, 2, 0, 1};
        const std::vector<std::vector<uint8_t>> plant = {{0, 1, 2, 3}, {3, 2, 0, 1}, {0, 1, 2, 3, 3, 2, 0, 1}};
        struct Case { int64_t span_lo, span_hi, thr; int fields; const char* what; };
        const int64_t F21 = 1 << 20, F32 = int64_t(1) << 31;
        const Case cases[] = {
            {-196608, 196608, F21 / 2, 3, "bmax - thr = 2^20 (21-bit field exactly full)"},
            {-196608, 196608, F21 - 1, 3, "thr = 2^20 - 1 (bias 0)"},
            {-196608, 196608, F21 / 2 - 1, 2, "bmax - thr = 2^20 + 1"},
            {-196608, 196608, F21, 2, "thr = 2^20"},
            {-402653184, 268435456, F32 / 4, 2, "bmax - thr = 2^31 (32-bit field exactly full)"},
            {-402653184, 268435456, F32 / 4 - 1, 0, "bmax - thr = 2^31 + 1"},
            {-402653184, 268435456, F32, 0, "thr = 2^31"},
        };
        for (const Case& k : cases) {
            std::vector<int32_t> w0(16, 1000), w1(16), w2(16);
            for (int c = 0; c < 4; ++c) { w0[4 * c + best[c]] = (int32_t)k.span_hi; w0[4 * c + worst[c]] = (int32_t)k.span_lo; }
            for (int i = 0; i < 16; ++i) { w1[i] = (int32_t)(rng() % 121) - 60; w2[i] = (int32_t)(rng() % 121) - 60; }
            int s1b = 0, s1w = 0, s2b = 0;
            for (int c = 0; c < 4; ++c) { s1b += w1[4 * c + best[c]]; s1w += w1[4 * c + worst[c]]; s2b += w2[4 * c + best[c]]; }
            w1[worst[0]] += s1b + 1 - s1w;  // slot 1: min_score on B, min_score + 1 on W
            const int64_t M = 4 * k.span_lo;
            const int64_t ms0 = M + k.thr;
            if (ms0 > INT32_MAX || ms0 < INT32_MIN) { printf("FAIL %s: min_score outside int32\n", k.what); ++bad; continue; }
            std::vector<tfbs_pattern> pats(3);
            const std::vector<int32_t>* ws[3] = {&w0, &w1, &w2};
            const int32_t ms[3] = {(int32_t)ms0, s1b, s2b - 1};
            for (int f = 0; f < 3; ++f) pats[f] = tfbs_pattern{ws[f]->data(), 4, ms[f], (uint16_t)(f + 1), 0, TFBS_PATTERN_PWM};
            CompiledPatterns cp;
            std::string err;
            int rc = compile_patterns(pats.data(), 3, 96 * 1024, 0, &cp, &err);
            if (k.fields == 0) {
                if (rc != TFBS_ERR_SCORE_RANGE) { printf("FAIL %s: accepted (rc %d, fields %u)\n", k.what, rc, cp.fields); ++bad; }
                else printf("ok %s: TFBS_ERR_SCORE_RANGE\n", k.what);
                continue;
            }
            if (rc != TFBS_OK || (int)cp.fields != k.fields) {
                printf("FAIL %s: rc %d, fields %u, expected %d\n", k.what, rc, cp.fields, k.fields);
                ++bad;
                continue;
            }
            bad += check(pats, 96 * 1024, 0, rng, k.what, plant);
        }
    }
    // error paths
    {
        CompiledPatterns cp;
        std::string err;
        std::vector<int32_t> w(4 * 33, 1);
        tfbs_pattern p{w.data(), 33, 0, 0, 0, TFBS_PATTERN_PWM};
        if (compile_patterns(&p, 1, 96 * 1024, 0, &cp, &err) != TFBS_ERR_INVALID_ARGUMENT) { printf("FAIL: 33 columns accepted\n"); ++bad; }
        tfbs_pattern e{nullptr, 0, 0, 0, 0, TFBS_PATTERN_PWM};
        if (compile_patterns(&e, 1, 96 * 1024, 0, &cp, &err) != TFBS_ERR_INVALID_ARGUMENT) { printf("FAIL: empty PWM accepted\n"); ++bad; }
        std::vector<int32_t> big(4 * 20);
        for (size_t i = 0; i < big.size(); ++i) big[i] = (i % 4 == 0) ? 2000000000 : -2000000000;
        tfbs_pattern g{big.data(), 20, 0, 0, 0, TFBS_PATTERN_PWM};
        if (compile_patterns(&g, 1, 96 * 1024, 0, &cp, &err) != TFBS_ERR_SCORE_RANGE) { printf("FAIL: score range not detected\n"); ++bad; }
    }
    printf(bad ? "FAILED\n" : "ALL OK\n");
    return bad ? 1 : 0;
}
