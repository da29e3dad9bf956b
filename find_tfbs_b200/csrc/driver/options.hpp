// options.hpp -- the reference's command line (main.rs:169-227) plus the driver's own options
// Host side of find-tfbs-b200 (see driver.cpp for the map); header-only, one translation unit.
#pragma once
#include "common.hpp"

namespace {

// ---------------------------------------------------------------------------------------------------------------
// options
// ---------------------------------------------------------------------------------------------------------------
struct Options {
    std::string chromosome, bcf, output, reference, pwm_file, threshold_dir, samples_file;
    std::string audit_file;  // --audit: threshold ties, truncated and overwritten haplotypes (tfbs_audit_block), tab-separated
    std::string attribution_file;  // --attribution: per written row, the configurations of records that change its count (tfbs_get_attribution)
    std::vector<std::string> beds, pwm_names;
    float pwm_threshold = 0;
    bool forward_only = false, tabix = false, verbose = false, has_samples = false, plain_text = false;
    uint32_t min_maf = 0, threads = 1, chunk = 0;  // chunk: merged regions per block (0 = automatic)
    std::string write_thresholds;  // --write_thresholds DIR: write <name>.thr for the PWMs of --pwm_file (exact DP), then exit
    std::vector<double> pvalues{1e-2, 1e-3, 5e-4, 1e-4, 1e-5};
    int compression_level = 3;  // zlib level of the BGZF blocks: the byte stream is not part of the contract (outputs are compared after gunzip)
    uint64_t after_position = 0;
    std::vector<int> devices{0};
    bool use_index = true;   // --no_index: ignore <bcf>.csi and scan the whole BCF
};

std::vector<std::string> split(const std::string& s, char sep) {
    std::vector<std::string> out;
    size_t p = 0;
    for (;;) {
        size_t q = s.find(sep, p);
        out.push_back(s.substr(p, q == std::string::npos ? std::string::npos : q - p));
        if (q == std::string::npos) break;
        p = q + 1;
    }
    return out;
}

void usage() {
    puts("find-tfbs-b200 1.0.1 (B200-native hot path)\n"
         "USAGE: find-tfbs-b200 --chromosome CHROM --input IN.bcf --output OUT.vcf.gz --reference REF.fa --bed A.bed[,B.bed]\n"
         "         --pwm_names NAME[,NAME] --pwm_file PWM.txt --pwm_threshold_directory DIR --pwm_threshold P\n"
         "         [--forward_only] [--threads N] [--min_maf N] [--after_position POS] [--samples FILE] [--tabix] [--verbose]\n"
         "         [--devices 0,1,...] [--chunk REGIONS_PER_BLOCK] [--plain] [--audit AUDIT.tsv] [--no_index] [--compression_level 1..9]\n"
         "         [--attribution ATTRIBUTION.tsv]\n"
         "       find-tfbs-b200 --write_thresholds DIR --pwm_file PWM.txt [--pwm_names NAME[,NAME]] [--pvalues P[,P]]   (exact .thr files)");
}

Options parse_args(int argc, char** argv) {
    Options o;
    std::map<std::string, std::string> kv;
    std::set<std::string> flags{"forward_only", "tabix", "verbose", "plain", "help", "no_index"};
    std::map<std::string, std::string> shorts{{"-c", "chromosome"}, {"-i", "input"}, {"-o", "output"}, {"-r", "reference"}, {"-b", "bed"},
                                              {"-p", "pwm_file"}, {"-f", "forward_only"}, {"-m", "min_maf"}, {"-s", "samples"},
                                              {"-z", "tabix"}, {"-v", "verbose"}};
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i], key, val;
        bool has_val = false;
        if (a.rfind("--", 0) == 0) {
            size_t eq = a.find('=');
            key = a.substr(2, eq == std::string::npos ? std::string::npos : eq - 2);
            if (eq != std::string::npos) { val = a.substr(eq + 1); has_val = true; }
        } else if (shorts.count(a)) key = shorts[a];
        else die("error: Found argument '" + a + "' which wasn't expected");
        if (flags.count(key)) { kv[key] = "1"; continue; }
        if (!has_val) {
            if (i + 1 >= argc) die("error: The argument '--" + key + "' requires a value");
            val = argv[++i];
        }
        kv[key] = val;
    }
    if (kv.count("help")) { usage(); exit(0); }
    if (kv.count("write_thresholds")) {  // threshold tooling: needs the PWM definitions only
        o.write_thresholds = kv["write_thresholds"];
        if (!kv.count("pwm_file")) { usage(); die("error: The following required argument was not provided: --pwm_file"); }
        o.pwm_file = kv["pwm_file"];
        if (kv.count("pwm_names")) o.pwm_names = split(kv["pwm_names"], ',');
        if (kv.count("pvalues")) {
            o.pvalues.clear();
            for (auto& t : split(kv["pvalues"], ',')) o.pvalues.push_back(atof(t.c_str()));
        }
        return o;
    }
    auto req = [&](const char* k) -> std::string {
        if (!kv.count(k)) { usage(); die(std::string("error: The following required argument was not provided: --") + k); }
        return kv[k];
    };
    o.chromosome = req("chromosome");
    o.bcf = req("input");
    o.output = req("output");
    o.reference = req("reference");
    o.beds = split(req("bed"), ',');
    o.pwm_names = split(req("pwm_names"), ',');
    o.pwm_file = req("pwm_file");
    o.threshold_dir = req("pwm_threshold_directory");
    {
        char* e = nullptr;
        std::string t = req("pwm_threshold");
        o.pwm_threshold = strtof(t.c_str(), &e);
        if (e == t.c_str() || *e) die("Cannot parse MAF");  // sic, main.rs:195
    }
    o.forward_only = kv.count("forward_only");
    o.tabix = kv.count("tabix");
    o.verbose = kv.count("verbose");
    o.plain_text = kv.count("plain");
    o.use_index = !kv.count("no_index");
    auto num = [&](const char* k, uint64_t dflt, const char* what) -> uint64_t {
        if (!kv.count(k)) return dflt;
        char* e = nullptr;
        unsigned long long v = strtoull(kv[k].c_str(), &e, 10);
        if (e == kv[k].c_str() || *e) die(what);
        return v;
    };
    o.min_maf = (uint32_t)num("min_maf", 0, "Cannot parse MAF");
    o.threads = (uint32_t)num("threads", 1, "Cannot parse thread number");
    if (kv.count("threads") && o.threads < 1) die("Wrong number of threads");
    o.after_position = num("after_position", 0, "Cannot parse after_position");
    o.chunk = (uint32_t)num("chunk", 0, "Cannot parse chunk");  // 0 = chosen from the cohort size once the BCF header is read
    o.compression_level = (int)std::min<uint64_t>(9, std::max<uint64_t>(1, num("compression_level", 3, "Cannot parse compression_level")));
    if (kv.count("samples")) { o.has_samples = true; o.samples_file = kv["samples"]; }
    if (kv.count("audit")) o.audit_file = kv["audit"];
    if (kv.count("attribution")) o.attribution_file = kv["attribution"];
    if (!o.audit_file.empty() && !o.attribution_file.empty()) die("error: --attribution cannot be used with --audit");
    if (kv.count("devices")) {
        o.devices.clear();
        for (auto& d : split(kv["devices"], ',')) o.devices.push_back(atoi(d.c_str()));
    }
    return o;
}

}  // namespace
