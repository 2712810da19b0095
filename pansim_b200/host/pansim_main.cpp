// pansim_main.cpp -- the `pansim` command line on top of libpansim_b200.so.
// C++ stand-in for the Rust host of pansim/src/main.rs (no Rust toolchain in this
// image): same 27 long flags and defaults (main.rs:21-151), same parsing quirks
// (sizes parsed as f64 then rounded, main.rs:155-167), same validation messages and
// exit code 0 on rejection (main.rs:194-247), same derived rates (main.rs:259-367),
// same call order per generation (main.rs:429-528) and the same six output files with
// Rust's `{}` float formatting. Host randomness (selection coefficients, initial rows,
// pair sampling) uses std::mt19937_64 in place of rand's StdRng.
#include <algorithm>
#include <charconv>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <map>
#include <random>
#include <string>
#include <vector>

#include "population.hpp"

namespace {

// Rust `{}` for f64: shortest round-trip digits, positional, "NaN"/"inf"
std::string fmt(double x)
{
    if (std::isnan(x)) return "NaN";
    if (std::isinf(x)) return x < 0 ? "-inf" : "inf";
    char buf[512];
    auto r = std::to_chars(buf, buf + sizeof buf, x, std::chars_format::fixed);
    return std::string(buf, r.ptr);
}

struct Flags {
    std::map<std::string, std::string> val;
    std::map<std::string, bool> sw;
};

const char *VALUE_FLAGS[] = {"pop_size", "core_size", "pan_genes", "core_genes", "avg_gene_freq", "n_gen",
                             "max_distances", "core_mu", "HR_rate", "HGT_rate", "rate_genes1", "rate_genes2",
                             "prop_genes2", "prop_positive", "pos_lambda", "neg_lambda", "seed", "outpref",
                             "threads", "genome_size_penalty", "competition_strength", "device", "gpus",
                             "ld_max_dist", "ld_bin_width", "ld_min_minor",        // extensions: --print_ld bins,
                             "gene_ld_bins", "gene_ld_min_minor",                  // --print_gene_ld histogram and genes,
                             "gene_accumulation_perms"};                           // --print_gene_accumulation orders
const char *SWITCH_FLAGS[] = {"print_dist", "print_matrices", "print_selection", "verbose", "no_control_genome_size",
                              "all_pairs", "print_diversity", "print_vcf", "print_ld", "print_genealogy",
                              "print_fasta", "print_snp_alignment", "print_gene_ld",
                              "print_gene_accumulation", "print_parsimony",
                              "print_nj"};                                    // extensions: all_pairs (every pair i < j in <outpref>.tsv),
                                                                              // print_diversity (<outpref>_diversity.tsv, <outpref>_core_sfs.txt),
                                                                              // print_vcf (<outpref>_core_genome.vcf),
                                                                              // print_ld (<outpref>_core_ld.tsv),
                                                                              // print_genealogy (<outpref>_genealogy.nwk, <outpref>_tmrca.tsv),
                                                                              // print_fasta (<outpref>_core_genome.fasta),
                                                                              // print_snp_alignment (<outpref>_core_snps.fasta, <outpref>_core_snps_fconst.txt),
                                                                              // print_gene_ld (<outpref>_gene_ld.tsv),
                                                                              // print_gene_accumulation (<outpref>_number_of_*.Rtab,
                                                                              //   <outpref>_gene_spectrum.txt, <outpref>_summary_statistics.txt),
                                                                              // print_parsimony (<outpref>_parsimony.tsv, <outpref>_core_site_changes.txt,
                                                                              //   <outpref>_gene_changes.txt, <outpref>_branch_changes.tsv),
                                                                              // print_nj (<outpref>_core_nj.nwk, <outpref>_acc_nj.nwk, <outpref>_nj_rf.tsv)

bool parse(int argc, char **argv, Flags &f)
{
    f.val = {{"pop_size", "1000"}, {"core_size", "1200000"}, {"pan_genes", "6000"}, {"core_genes", "2000"},
             {"avg_gene_freq", "0.5"}, {"n_gen", "100"}, {"max_distances", "100000"}, {"core_mu", "0.05"},
             {"HR_rate", "0.05"}, {"HGT_rate", "0.05"}, {"rate_genes1", "1.0"}, {"rate_genes2", "1000.0"},
             {"prop_genes2", "0.1"}, {"prop_positive", "-0.1"}, {"pos_lambda", "10.0"}, {"neg_lambda", "10.0"},
             {"seed", "0"}, {"outpref", "distances"}, {"threads", "1"}, {"genome_size_penalty", "0.99"},
             {"competition_strength", "0.0"}, {"device", "0"}, {"gpus", "1"},
             {"ld_max_dist", "10000"}, {"ld_bin_width", "100"}, {"ld_min_minor", "1"},
             {"gene_ld_bins", "20"}, {"gene_ld_min_minor", "1"}, {"gene_accumulation_perms", "100"}};
    for (int i = 1; i < argc; i++) {
        std::string a = argv[i];
        if (a == "--help" || a == "-h") {
            std::printf("pansim 0.1.0 (B200 build)\nRuns Wright-Fisher simulation, simulating neutral core genome "
                        "evolution and two-speed accessory genome evolution.\n\nOPTIONS:\n");
            for (const char *n : VALUE_FLAGS) std::printf("    --%s <%s> [default: %s]\n", n, n, f.val[n].c_str());
            for (const char *n : SWITCH_FLAGS) std::printf("    --%s\n", n);
            return false;
        }
        if (a.rfind("--", 0) != 0) { std::fprintf(stderr, "error: unexpected argument '%s'\n", a.c_str()); std::exit(2); }
        std::string name = a.substr(2), value;
        const size_t eq = name.find('=');
        bool has_value = false;
        if (eq != std::string::npos) { value = name.substr(eq + 1); name = name.substr(0, eq); has_value = true; }
        bool is_switch = false;
        for (const char *n : SWITCH_FLAGS) if (name == n) is_switch = true;
        if (is_switch) { f.sw[name] = true; continue; }
        if (!f.val.count(name)) { std::fprintf(stderr, "error: unknown flag '--%s'\n", name.c_str()); std::exit(2); }
        if (!has_value) {
            if (i + 1 >= argc) { std::fprintf(stderr, "error: flag '--%s' needs a value\n", name.c_str()); std::exit(2); }
            value = argv[++i];
        }
        f.val[name] = value;
    }
    return true;
}

double as_f64(const Flags &f, const char *n) { return std::strtod(f.val.at(n).c_str(), nullptr); }
size_t as_rounded(const Flags &f, const char *n) { return (size_t)std::llround(as_f64(f, n)); }   // main.rs:155-167

}  // namespace

void pansim::Populations::write(const std::string &outpref)
{
    const size_t N = cfg_.pop_size, L = cfg_.core_size, G = cfg_.pan_size;
    {
        std::ofstream f(outpref + "_core_genome.csv", std::ios::binary);
        const uint32_t step = (uint32_t)std::max<size_t>(1, (64u << 20) / std::max<size_t>(1, 2 * L));
        std::vector<char> buf((size_t)step * 2 * L);
        for (uint32_t r0 = 0; r0 < N; r0 += step) {
            const uint32_t r1 = (uint32_t)std::min<size_t>(N, r0 + step);
            gcheck(pansim_group_export_core_csv(grp_, r0, r1, buf.data()));   // one GPU: pinned double-buffered stream (pansim_export_core_csv)
            f.write(buf.data(), (std::streamsize)((size_t)(r1 - r0) * 2 * L));
        }
    }
    std::vector<uint8_t> acc(N * G);
    gcheck(pansim_group_download_acc(grp_, acc.data()));
    std::ofstream f(outpref + "_pangenome.csv");
    for (size_t r = 0; r < N; r++) {
        std::string line;
        for (uint32_t k = 0; k < cfg_.core_genes; k++) { if (!line.empty()) line += ','; line += '1'; }   // population.rs:891
        for (size_t g = 0; g < G; g++) { if (!line.empty()) line += ','; line += (char)('0' + acc[r * G + g]); }
        f << line << "\n";
    }
}

int main(int argc, char **argv)
{
    Flags fl;
    if (!parse(argc, argv, fl)) return 0;
    const size_t pop_size = as_rounded(fl, "pop_size"), core_size = as_rounded(fl, "core_size");
    const size_t pan_genes = as_rounded(fl, "pan_genes"), core_genes = as_rounded(fl, "core_genes");
    double avg_gene_freq = as_f64(fl, "avg_gene_freq");
    const double HR_rate = as_f64(fl, "HR_rate"), HGT_rate = as_f64(fl, "HGT_rate");
    const int n_gen = (int)std::llround(as_f64(fl, "n_gen"));
    const std::string outpref = fl.val["outpref"];
    const size_t max_distances = std::strtoull(fl.val["max_distances"].c_str(), nullptr, 10);
    const double core_mu = as_f64(fl, "core_mu"), rate_genes1 = as_f64(fl, "rate_genes1"), rate_genes2 = as_f64(fl, "rate_genes2");
    const double prop_genes2 = as_f64(fl, "prop_genes2"), prop_positive = as_f64(fl, "prop_positive");
    const double pos_lambda = as_f64(fl, "pos_lambda"), neg_lambda = as_f64(fl, "neg_lambda");
    const uint64_t seed = std::strtoull(fl.val["seed"].c_str(), nullptr, 10);
    const bool verbose = fl.sw["verbose"], print_dist = fl.sw["print_dist"], print_matrices = fl.sw["print_matrices"];
    const bool all_pairs = fl.sw["all_pairs"], print_diversity = fl.sw["print_diversity"], print_vcf = fl.sw["print_vcf"];
    const bool print_ld = fl.sw["print_ld"], print_genealogy = fl.sw["print_genealogy"];
    const bool print_fasta = fl.sw["print_fasta"], print_snp_alignment = fl.sw["print_snp_alignment"];
    const pansim_ld_params ld_params = {(uint32_t)std::strtoul(fl.val["ld_max_dist"].c_str(), nullptr, 10),
                                        (uint32_t)std::strtoul(fl.val["ld_bin_width"].c_str(), nullptr, 10),
                                        (uint32_t)std::strtoul(fl.val["ld_min_minor"].c_str(), nullptr, 10)};
    const bool print_gene_ld = fl.sw["print_gene_ld"];
    const bool print_gene_accumulation = fl.sw["print_gene_accumulation"];
    const bool print_parsimony = fl.sw["print_parsimony"];
    const bool print_nj = fl.sw["print_nj"];
    const uint32_t gene_accumulation_perms = (uint32_t)std::strtoul(fl.val["gene_accumulation_perms"].c_str(), nullptr, 10);
    const pansim_gene_ld_params gene_ld_params = {(uint32_t)std::strtoul(fl.val["gene_ld_bins"].c_str(), nullptr, 10),
                                                  (uint32_t)std::strtoul(fl.val["gene_ld_min_minor"].c_str(), nullptr, 10)};
    const int n_gpus = std::max(1, std::atoi(fl.val["gpus"].c_str()));       // extension: column shards over N devices of the box
    const bool print_selection = fl.sw["print_selection"], no_control = fl.sw["no_control_genome_size"];
    const double genome_size_penalty = as_f64(fl, "genome_size_penalty"), competition_strength = as_f64(fl, "competition_strength");

    // ---- validation, main.rs:194-247 (print and exit 0) ----
    if (core_genes > pan_genes) { std::printf("core_genes must be less than or equal to pan_size\n"); return 0; }
    if (HR_rate < 0.0 || HGT_rate < 0.0) { std::printf("HR_rate and HGT_rate must be above 0.0\nHR_rate: %s\nHGT_rate: %s\n", fmt(HR_rate).c_str(), fmt(HGT_rate).c_str()); return 0; }
    if (pos_lambda <= 0.0 || neg_lambda <= 0.0) { std::printf("pos_lambda and neg_lambda must be above 0.0\npos_lambda: %s\nneg_lambda: %s\n", fmt(pos_lambda).c_str(), fmt(neg_lambda).c_str()); return 0; }
    if (rate_genes1 < 0.0 || rate_genes2 < 0.0) { std::printf("rate_genes1 and rate_genes2 must be >= 0\nrate_genes1: %s\nrate_genes2: %s\n", fmt(rate_genes1).c_str(), fmt(rate_genes2).c_str()); return 0; }
    if (prop_genes2 < 0.0 || prop_genes2 > 1.0) { std::printf("prop_genes2 must be 0.0 <= prop_genes2 <= 1.0\nprop_genes2: %s\n", fmt(prop_genes2).c_str()); return 0; }
    if (pop_size < 1 || core_size < 1 || pan_genes < 1 || n_gen < 1 || max_distances < 1) {
        std::printf("pop_size, core_size, pan_genes, n_gen and max_distances must all be above 1\npop_size: %zu\ncore_size: %zu\npan_genes: %zu\nn_gen: %d\nmax_distances: %zu\n", pop_size, core_size, pan_genes, n_gen, max_distances);
        return 0;
    }
    if (core_mu < 0.0 || core_mu > 1.0) { std::printf("core_mu must be between 0.0 and 1.0\ncore_mu: %s\n", fmt(core_mu).c_str()); return 0; }
    if (avg_gene_freq <= 0.0 || avg_gene_freq > 1.0) { std::printf("avg_gene_freq must be above 0.0 and below or equal to 1.0\navg_gene_freq: %s\n", fmt(avg_gene_freq).c_str()); return 0; }

    // ---- derived parameters, main.rs:259-287, 333-367 ----
    const size_t pan_size = pan_genes - core_genes;
    const double core_prop = (double)core_genes / (double)pan_genes, acc_prop = 1.0 - core_prop;
    avg_gene_freq = (avg_gene_freq - core_prop) / acc_prop;
    if (avg_gene_freq < 0.0) avg_gene_freq = 0.0;
    if (verbose) std::printf("avg_gene_freq adjusted to %s\n", fmt(avg_gene_freq).c_str());
    const int32_t avg_gene_num = (int32_t)std::llround(avg_gene_freq * (double)pan_size);
    const double n_core_mutations = std::ceil((double)core_size * core_mu);
    const double n_recombinations_core = std::round(n_core_mutations * HR_rate);
    const double n_recombinations_pan_total = std::round(n_core_mutations * HGT_rate);
    const size_t num_gene1_sites = (size_t)std::llround((double)pan_size * (1.0 - prop_genes2));
    const size_t num_gene2_sites = pan_size - num_gene1_sites;
    const double prop_gene1_sites = (double)num_gene1_sites / (double)pan_size, prop_gene2_sites = 1.0 - prop_gene1_sites;

    pansim_config cfg;
    pansim_config_init(&cfg);
    cfg.device = std::atoi(fl.val["device"].c_str());
    cfg.pop_size = (uint32_t)pop_size; cfg.pan_size = (uint32_t)pan_size; cfg.core_size = core_size;
    cfg.core_genes = (uint32_t)core_genes;
    uint32_t c = 0;
    if (num_gene1_sites > 0) {
        cfg.comp_lo[c] = 0; cfg.comp_hi[c] = (uint32_t)num_gene1_sites;
        cfg.acc_mut_mean[c] = rate_genes1 * (double)num_gene1_sites;
        cfg.hgt_mean[c] = HGT_rate > 0.0 ? n_recombinations_pan_total * prop_gene1_sites : 0.0;
        c++;
    }
    if (num_gene1_sites < pan_size) {
        cfg.comp_lo[c] = (uint32_t)num_gene1_sites; cfg.comp_hi[c] = (uint32_t)pan_size;
        cfg.acc_mut_mean[c] = rate_genes2 * (double)num_gene2_sites;
        cfg.hgt_mean[c] = HGT_rate > 0.0 ? n_recombinations_pan_total * prop_gene2_sites : 0.0;
        c++;
    }
    cfg.n_compartments = c;
    cfg.core_mut_mean = n_core_mutations;
    cfg.hr_mean = HR_rate > 0.0 ? n_recombinations_core : 0.0;
    cfg.avg_gene_num = avg_gene_num; cfg.no_control_genome_size = no_control ? 1 : 0;
    cfg.genome_size_penalty = genome_size_penalty; cfg.competition_strength = competition_strength; cfg.seed = seed;

    // ---- host-side random setup (main.rs:289-319, 372-427) ----
    std::mt19937_64 rng(seed);
    std::uniform_real_distribution<double> uni(0.0, 1.0);
    std::vector<double> selection(pan_size, 0.0);
    if (prop_positive >= 0.0) {
        std::exponential_distribution<double> epos(pos_lambda), eneg(neg_lambda);
        for (size_t i = 0; i < pan_size; i++) {
            if (uni(rng) <= prop_positive) selection[i] = epos(rng);
            else { double s = eneg(rng); while (s > 1.0) s = eneg(rng); selection[i] = -1.0 * s; }
        }
    }
    if (print_selection) {
        std::ofstream f(outpref + "_selection.tsv");
        for (size_t i = 0; i < pan_size; i++) f << (i ? "\n" : "") << fmt(selection[i]);
        f << "\n";
    }
    std::vector<uint8_t> core_row(core_size), acc_row(pan_size);
    for (auto &b : core_row) b = (uint8_t)(1u << (rng() & 3));
    for (auto &b : acc_row) b = uni(rng) < avg_gene_freq ? 1 : 0;
    std::vector<uint32_t> range1(max_distances), range2(max_distances);
    if (pop_size < 2) { std::fprintf(stderr, "pansim: pop_size must be >= 2 to sample pairs\n"); return 101; }
    for (auto &v : range1) v = (uint32_t)(rng() % pop_size);
    for (size_t k = 0; k < max_distances; k++) {
        uint32_t e = (uint32_t)(rng() % (pop_size - 1));
        if (e >= range1[k]) e += 1;
        range2[k] = e;
    }

    try {
        pansim::Populations pops(cfg, n_gpus);
        pops.set_initial(core_row, acc_row);
        pops.set_selection(selection);
        if (print_genealogy || print_parsimony || print_nj) pops.enable_genealogy((uint32_t)n_gen);   // extension: after set_initial, which clears the record
        std::vector<double> avg_core(n_gen, 0.0), avg_acc(n_gen, 0.0), std_core(n_gen, 0.0), std_acc(n_gen, 0.0);
        std::vector<double> core_d, acc_d;
        std::vector<pansim_diversity> diversity;
        auto last_generation_outputs = [&]() {                              // main.rs:467-499
            std::ofstream f(outpref + ".tsv");
            if (all_pairs) {
                // every pair i < j in (i, j) order, row blocks of about 4 million pairs
                std::string line;
                pops.all_pairs(4000000, [&](double c_, double a_) { f << fmt(c_) << "\t" << fmt(a_) << "\n"; });
            } else {
                pops.pairwise_distances(range1, range2, core_d, acc_d);
                for (size_t k = 0; k < max_distances; k++) f << fmt(core_d[k]) << "\t" << fmt(acc_d[k]) << "\n";
            }
            std::ofstream g(outpref + "_freqs.txt");
            for (double x : pops.gene_frequencies()) g << fmt(x) << "\n";
        };
        // Nothing has to come back between generations unless --verbose asks for it: the run is one
        // device-resident batch (same states). With --print_dist the batch also makes the distance pass and
        // its mean / standard deviation on the device every generation (pansim_run_generations_stats).
        const bool device_loop = !verbose;
        int first_host_gen = 0;
        if (device_loop) {
            if (print_diversity) {                                          // one batch: reduction (+ --print_dist pass) per generation
                std::vector<double> st;
                const std::vector<uint32_t> none;
                diversity = pops.run_generations_diversity(0, (uint32_t)n_gen, print_dist ? range1 : none, print_dist ? range2 : none, st);
                for (int j = 0; j < n_gen && print_dist; j++) { avg_core[j] = st[4 * j]; std_core[j] = st[4 * j + 1]; avg_acc[j] = st[4 * j + 2]; std_acc[j] = st[4 * j + 3]; }
            } else if (print_dist) {
                const std::vector<double> st = pops.run_generations_stats(0, (uint32_t)n_gen, range1, range2);
                for (int j = 0; j < n_gen; j++) { avg_core[j] = st[4 * j]; std_core[j] = st[4 * j + 1]; avg_acc[j] = st[4 * j + 2]; std_acc[j] = st[4 * j + 3]; }
            } else {
                pops.run_generations(0, (uint32_t)n_gen);
            }
            first_host_gen = n_gen;
            last_generation_outputs();
        }
        for (int j = first_host_gen; j < n_gen; j++) {
            pops.step((uint32_t)j);                                         // main.rs:435-464
            if (print_diversity) diversity.push_back(pops.core_diversity());
            if (j == n_gen - 1) last_generation_outputs();
            if (print_dist) {                                               // main.rs:502-519
                if (j != n_gen - 1 || all_pairs) pops.pairwise_distances(range1, range2, core_d, acc_d);
                auto sc = pansim::standard_deviation(core_d), sa = pansim::standard_deviation(acc_d);
                std_core[j] = sc.first; avg_core[j] = sc.second; std_acc[j] = sa.first; avg_acc[j] = sa.second;
            }
            if (verbose) {                                                  // main.rs:522-526
                std::printf("Finished gen: %d\n", j + 1);
                std::printf("avg_gene_freq: %s\n", fmt(pops.calc_gene_freq()).c_str());
            }
        }
        if (print_dist) {                                                   // main.rs:531-548
            std::ofstream f(outpref + "_per_gen.tsv");
            for (int j = 0; j < n_gen; j++)
                f << fmt(avg_core[j]) << "\t" << fmt(std_core[j]) << "\t" << fmt(avg_acc[j]) << "\t" << fmt(std_acc[j]) << "\n";
        }
        if (print_diversity) {                                              // extension: core-genome diversity
            std::vector<uint64_t> sfs;
            pops.core_diversity(&sfs);
            std::ofstream f(outpref + "_diversity.tsv");
            for (const pansim_diversity &d : diversity) {
                double st[3];
                pansim_diversity_stats(&d, (uint32_t)pop_size, st);
                f << d.segregating << "\t" << d.multiallelic << "\t" << fmt(st[0]) << "\t" << fmt(st[1]) << "\t" << fmt(st[2]) << "\n";
            }
            std::ofstream g(outpref + "_core_sfs.txt");
            for (uint64_t x : sfs) g << x << "\n";
        }
        if (print_matrices) pops.write(outpref);                            // main.rs:550-553
        if (print_vcf) pops.write_core_vcf(outpref + "_core_genome.vcf");   // extension: the last generation as VCF
        if (print_ld) {                                                     // extension: LD of the last generation by distance
            std::ofstream f(outpref + "_core_ld.tsv");
            const std::vector<pansim_ld_bin> bins = pops.core_ld(ld_params);
            for (size_t b = 0; b < bins.size(); b++) {
                const uint64_t lo = (uint64_t)b * ld_params.bin_width + 1, hi = std::min<uint64_t>(lo + ld_params.bin_width - 1, ld_params.max_dist);
                f << lo << "\t" << hi << "\t" << bins[b].pairs << "\t" << bins[b].four_gamete << "\t" << fmt(pansim_ld_mean_r2(&bins[b])) << "\n";
            }
        }
        if (print_genealogy) {                                              // extension: the genealogy of the last generation
            std::ofstream(outpref + "_genealogy.nwk", std::ios::binary) << pops.newick(pops.genealogy());
            // one TMRCA per line of <outpref>.tsv: the sampled pairs, or every pair i < j in (i, j) order by row blocks
            std::ofstream f(outpref + "_tmrca.tsv");
            auto put = [&](const std::vector<uint32_t> &t) { for (uint32_t x : t) f << x << "\n"; };
            if (!all_pairs) {
                put(pops.tmrca(range1, range2));
            } else {
                std::vector<uint32_t> ii, jj;
                for (uint32_t i = 0; i + 1 < (uint32_t)pop_size; i++) {
                    for (uint32_t j = i + 1; j < (uint32_t)pop_size; j++) { ii.push_back(i); jj.push_back(j); }
                    if (ii.size() >= 4000000 || i + 2 == (uint32_t)pop_size) { put(pops.tmrca(ii, jj)); ii.clear(); jj.clear(); }
                }
            }
        }
        if (print_fasta) pops.write_core_fasta(outpref + "_core_genome.fasta", false);   // extension: the last generation as FASTA
        if (print_snp_alignment) {                                          // extension: its polymorphic columns, constant sites for -fconst
            uint64_t consts[4];
            pops.write_core_fasta(outpref + "_core_snps.fasta", true, consts);
            std::ofstream(outpref + "_core_snps_fconst.txt") << consts[0] << "," << consts[1] << "," << consts[2] << "," << consts[3] << "\n";
        }
        if (print_gene_ld) {                                                // extension: linkage of the accessory genes by class
            std::vector<uint64_t> hist;
            const std::array<pansim_gene_ld_class, 3> cls = pops.gene_ld(gene_ld_params, &hist);
            const char *label[3] = {"0-0", "0-1", "1-1"};
            std::ofstream f(outpref + "_gene_ld.tsv");
            for (int k = 0; k < 3; k++) {
                f << label[k] << "\t" << cls[k].ld.pairs << "\t" << cls[k].ld.four_gamete << "\t" << cls[k].associated << "\t"
                  << cls[k].dissociated << "\t" << fmt(pansim_ld_mean_r2(&cls[k].ld));
                for (uint32_t b = 0; b < gene_ld_params.r2_bins; b++) f << "\t" << hist[(size_t)k * gene_ld_params.r2_bins + b];
                f << "\n";
            }
        }
        if (print_gene_accumulation) {                                      // extension: Roary's pangenome summaries
            const auto acc = pops.gene_accumulation(seed, gene_accumulation_perms);
            const size_t N = pop_size;
            const std::pair<const char *, const std::vector<uint32_t> *> curves[4] = {
                {"genes_in_pan_genome", &acc.pan}, {"conserved_genes", &acc.core}, {"new_genes", &acc.new_genes},
                {"unique_genes", &acc.unique}};
            for (const auto &c : curves) {
                std::ofstream f(outpref + "_number_of_" + c.first + ".Rtab");
                for (size_t p = 0; p < gene_accumulation_perms; p++)
                    for (size_t k = 0; k < N; k++) f << (*c.second)[p * N + k] << (k + 1 < N ? "\t" : "\n");
            }
            const std::vector<uint64_t> spectrum = pops.gene_spectrum();
            {
                std::ofstream f(outpref + "_gene_spectrum.txt");
                for (uint64_t x : spectrum) f << x << "\n";
            }
            uint64_t cls[5];
            pansim_pangenome_classes(spectrum.data(), (uint32_t)N, cls);
            const char *label[5] = {"Core genes\t(99% <= strains <= 100%)", "Soft core genes\t(95% <= strains < 99%)",
                                    "Shell genes\t(15% <= strains < 95%)", "Cloud genes\t(0% <= strains < 15%)",
                                    "Total genes\t(0% <= strains <= 100%)"};
            std::ofstream f(outpref + "_summary_statistics.txt");
            for (int k = 0; k < 5; k++) f << label[k] << "\t" << cls[k] << "\n";
        }
        if (print_parsimony) {                                              // extension: parsimony on the true genealogy
            const std::vector<pansim_genealogy_node> nodes = pops.genealogy();
            const size_t n = nodes.size();
            std::vector<uint32_t> parent(n), first(n, (uint32_t)pop_size), below(n, 0);
            for (size_t k = 0; k < n; k++) parent[k] = nodes[k].parent;
            const auto core = pops.core_parsimony(parent);
            const auto genes = pops.gene_parsimony(parent);
            {
                std::ofstream f(outpref + "_parsimony.tsv");
                const std::pair<const char *, const pansim_parsimony *> rows[2] = {{"core", &core.summary}, {"genes", &genes.summary}};
                for (const auto &r : rows) {
                    const pansim_parsimony &q = *r.second;
                    double ci = 0.0, ri = 0.0;
                    pansim_parsimony_indices(&q, &ci, &ri);
                    f << r.first << "\t" << q.characters << "\t" << q.variable << "\t" << q.tree_length << "\t" << q.min_changes
                      << "\t" << q.max_changes << "\t" << q.homoplastic << "\t" << fmt(ci) << "\t" << fmt(ri) << "\n";
                }
            }
            {
                std::ofstream f(outpref + "_core_site_changes.txt");
                for (uint32_t x : core.site_changes) f << x << "\n";
            }
            {
                std::ofstream f(outpref + "_gene_changes.txt");
                for (uint32_t x : genes.gene_changes) f << x << "\n";
            }
            // (first leaf, leaves below) of every node: the key of a clade in _genealogy.nwk, whose internal nodes
            // carry no label
            for (size_t k = 0; k < (size_t)pop_size && k < n; k++) { first[k] = (uint32_t)k; below[k] = 1; }
            for (size_t k = 0; k + 1 < n; k++) {
                first[parent[k]] = std::min(first[parent[k]], first[k]);
                below[parent[k]] += below[k];
            }
            std::ofstream f(outpref + "_branch_changes.tsv");
            for (size_t k = 0; k + 1 < n; k++)
                f << k << "\t" << parent[k] << "\t" << first[k] << "\t" << below[k] << "\t" << nodes[parent[k]].time - nodes[k].time
                  << "\t" << core.branch_changes[k] << "\t" << genes.gains[k] << "\t" << genes.losses[k] << "\n";
        }
        if (print_nj) {                                                     // extension: NJ trees against the true genealogy
            const std::vector<pansim_genealogy_node> nodes = pops.genealogy();
            std::vector<uint32_t> gparent(nodes.size());
            for (size_t k = 0; k < nodes.size(); k++) gparent[k] = nodes[k].parent;
            std::ofstream rf(outpref + "_nj_rf.tsv");
            for (const char *metric : {"core", "acc"}) {
                const auto t = pops.nj_tree(metric[0] == 'c' ? 0 : 1);
                std::ofstream(outpref + "_" + metric + "_nj.nwk") << pops.tree_newick(t.parent, t.length);
                const auto s = pops.compare_splits(t.parent, gparent);
                const uint64_t total = s[0] + s[1], d = total - 2 * s[2];
                rf << metric << "\t" << s[0] << "\t" << s[1] << "\t" << s[2] << "\t" << d << "\t"
                   << fmt(total ? (double)d / (double)total : std::nan("")) << "\n";
            }
        }
    } catch (const pansim::Error &e) {
        // the reference aborts with a panic message (exit status 101)
        std::fprintf(stderr, "pansim: %s\n", e.what());
        return 101;
    }
    return 0;
}
