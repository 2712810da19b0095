// population.hpp -- C++ host-side mirror of the reference's `Population` API
// (pansim/src/population.rs) over the C ABI of include/pansim_b200.h.
//
// The reference keeps two Population objects (core_genome, pan_genome) that are
// always advanced together with the same parent vector (main.rs:442-464); here one
// `Populations` object owns both of them, on one GPU or column-sharded over several
// (pansim_group: one process, NCCL inside the library, `pansim --gpus N`). Method names, argument
// meaning and error behaviour follow population.rs; errors surface as
// pansim::Error (the reference panics via unwrap()).
#pragma once
#include <array>
#include <cmath>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/pansim_b200.h"

namespace pansim {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string &m) : std::runtime_error(m), code(c) {}
};

// population.rs:87-94: returns (std, mean); population variance, sequential sums
inline std::pair<double, double> standard_deviation(const std::vector<double> &v)
{
    double sum = 0.0;
    for (double x : v) sum += x;
    const double mean = sum / (double)v.size();
    double ss = 0.0;
    for (double x : v) ss += (x - mean) * (x - mean);
    return {std::sqrt(ss / (double)v.size()), mean};
}

// population.rs:154-162
inline char int_to_base(uint8_t n)
{
    switch (n) { case 1: return 'A'; case 2: return 'C'; case 4: return 'G'; case 8: return 'T'; default: return 'N'; }
}

class Populations {
public:
    explicit Populations(const pansim_config &cfg, int n_gpus = 1) : cfg_(cfg)
    {
        std::vector<int> devs;
        for (int i = 0; i < n_gpus; i++) devs.push_back(cfg.device + i);
        const int rc = pansim_group_create(&cfg_, n_gpus, devs.data(), &grp_);
        if (rc != PANSIM_OK) throw Error(rc, pansim_group_last_error(nullptr));
        ctx_ = pansim_group_ctx(grp_, 0);
    }
    ~Populations() { pansim_group_destroy(grp_); }
    int n_gpus() const { return pansim_group_size(grp_); }
    Populations(const Populations &) = delete;
    Populations &operator=(const Populations &) = delete;

    // Population::new x2 (population.rs:181-242): every row starts as the given row
    void set_initial(const std::vector<uint8_t> &core_row_onehot, const std::vector<uint8_t> &acc_row)
    {
        gcheck(pansim_group_set_initial(grp_, core_row_onehot.data(), acc_row.data()));
    }
    void set_selection(const std::vector<double> &s) { gcheck(pansim_group_set_selection(grp_, s.data())); }

    // population.rs:753-784 (accessory population)
    std::vector<double> average_distance()
    {
        single("average_distance");
        std::vector<double> out(cfg_.pop_size);
        check(pansim_average_distance(ctx_, out.data()));
        return out;
    }
    // population.rs:270-448
    std::vector<uint32_t> sample_indices(uint32_t gen, const std::vector<double> &avg_pairwise_dists)
    {
        single("sample_indices");
        std::vector<uint32_t> out(cfg_.pop_size);
        check(pansim_sample_indices(ctx_, gen, avg_pairwise_dists.empty() ? nullptr : avg_pairwise_dists.data(), out.data()));
        return out;
    }
    // population.rs:450-465 for both populations
    void next_generation(const std::vector<uint32_t> &parents) { single("next_generation"); check(pansim_next_generation(ctx_, parents.data())); }
    // main.rs:445-464 in one fused pass (next_generation + mutate_alleles + recombine, both populations)
    void step_with_parents(uint32_t gen, const std::vector<uint32_t> &parents)
    {
        single("step_with_parents");
        check(pansim_step_with_parents(ctx_, gen, parents.data()));
    }
    // main.rs:435-464 entirely on the device
    void step(uint32_t gen) { gcheck(pansim_group_run_generations(grp_, gen, 1)); }

    // population.rs:787-837 for both populations: f64 distances formed on the host from
    // the integer counts with the reference's own expressions (:822, :828-830)
    void pairwise_distances(const std::vector<uint32_t> &range1, const std::vector<uint32_t> &range2,
                            std::vector<double> &core_out, std::vector<double> &acc_out)
    {
        const size_t P = range1.size();
        std::vector<uint32_t> cd(P), in(P), un(P);
        gcheck(pansim_group_pair_counts(grp_, range1.data(), range2.data(), P, cd.data(), in.data(), un.data()));
        core_out.resize(P);
        acc_out.resize(P);
        for (size_t k = 0; k < P; k++) {
            core_out[k] = pansim_core_distance(cd[k], cfg_.core_size);
            acc_out[k] = pansim_acc_distance(in[k], un[k], cfg_.core_genes);
        }
    }
    // (extension, BASELINE config 5) exact all-pairs mode: `sink(core_distance, acc_distance)` is called for
    // every pair i < j in (i, j) order. Row blocks of about chunk_pairs pairs; over several GPUs the partial
    // core counts of a block are reduce-scattered while the next block is computed (pansim_group_all_pairs).
    template <typename Sink>
    void all_pairs(size_t chunk_pairs, Sink &&sink)
    {
        struct Ctx { Populations *self; Sink *sink; } u{this, &sink};
        auto cb = [](void *user, uint32_t, uint32_t, size_t n, const uint32_t *cd, const uint32_t *in, const uint32_t *un) -> int {
            Ctx *x = static_cast<Ctx *>(user);
            const pansim_config &cf = x->self->cfg_;
            for (size_t k = 0; k < n; k++) (*x->sink)(pansim_core_distance(cd[k], cf.core_size), pansim_acc_distance(in[k], un[k], cf.core_genes));
            return 0;
        };
        gcheck(pansim_group_all_pairs(grp_, chunk_pairs, cb, &u));
    }
    // main.rs:429-519 under --print_dist as one device-resident batch: per generation (avg_core, std_core, avg_acc, std_acc)
    std::vector<double> run_generations_stats(uint32_t gen0, uint32_t n, const std::vector<uint32_t> &range1,
                                              const std::vector<uint32_t> &range2)
    {
        std::vector<double> out((size_t)n * 4);
        gcheck(pansim_group_run_generations_stats(grp_, gen0, n, range1.data(), range2.data(), range1.size(), out.data()));
        return out;
    }
    // main.rs:435-464 for generations gen0 .. gen0+n-1 as one device-resident batch
    void run_generations(uint32_t gen0, uint32_t n) { gcheck(pansim_group_run_generations(grp_, gen0, n)); }
    // (extension) the same batch with the core-genome diversity reduction after every generation; with pairs
    // (range1 non-empty) also the --print_dist statistics, stats_out[n*4] as run_generations_stats gives them
    std::vector<pansim_diversity> run_generations_diversity(uint32_t gen0, uint32_t n, const std::vector<uint32_t> &range1,
                                                            const std::vector<uint32_t> &range2, std::vector<double> &stats_out)
    {
        std::vector<pansim_diversity> out(n);
        stats_out.assign(range1.empty() ? 0 : (size_t)n * 4, 0.0);
        gcheck(pansim_group_run_generations_diversity(grp_, gen0, n, range1.data(), range2.data(), range1.size(),
                                                      stats_out.empty() ? nullptr : stats_out.data(), out.data()));
        return out;
    }
    // (extension) core-genome diversity of the current state over the whole alignment; sfs [N+1] if non-null
    pansim_diversity core_diversity(std::vector<uint64_t> *sfs = nullptr)
    {
        pansim_diversity d;
        if (sfs) sfs->assign((size_t)cfg_.pop_size + 1, 0);
        gcheck(pansim_group_core_diversity(grp_, &d, sfs ? sfs->data() : nullptr));
        return d;
    }
    // population.rs:840-863: accessory gene frequencies, then core_genes x 1.0
    std::vector<double> gene_frequencies()
    {
        std::vector<uint32_t> counts(cfg_.pan_size);
        gcheck(pansim_group_gene_counts(grp_, counts.data()));
        std::vector<double> f;
        f.reserve(cfg_.pan_size + cfg_.core_genes);
        for (uint32_t c : counts) f.push_back((double)c / (double)cfg_.pop_size);
        for (uint32_t k = 0; k < cfg_.core_genes; k++) f.push_back(1.0);
        return f;
    }
    // population.rs:244-268
    double calc_gene_freq()
    {
        std::vector<uint8_t> acc((size_t)cfg_.pop_size * cfg_.pan_size);
        gcheck(pansim_group_download_acc(grp_, acc.data()));
        double sum = 0.0;
        for (uint32_t r = 0; r < cfg_.pop_size; r++) {
            size_t s = 0;
            for (uint32_t g = 0; g < cfg_.pan_size; g++) s += acc[(size_t)r * cfg_.pan_size + g];
            sum += (double)s / (double)cfg_.pan_size;
        }
        return sum / (double)cfg_.pop_size;
    }
    // population.rs:865-897 `write` for both populations
    void write(const std::string &outpref);
    // (extension) the core alignment as VCF against the initial row, all shards in one file; bytes written
    uint64_t write_core_vcf(const std::string &path)
    {
        uint64_t n = 0;
        gcheck(pansim_group_write_core_vcf(grp_, path.c_str(), &n));
        return n;
    }
    // (extension) the core alignment as FASTA, every site or (snps_only) the polymorphic columns, all shards in one
    // file; the constant-site counts by letter go to const_counts[4] if given; bytes written
    uint64_t write_core_fasta(const std::string &path, bool snps_only, uint64_t *const_counts = nullptr)
    {
        uint64_t n = 0;
        gcheck(pansim_group_write_core_fasta(grp_, path.c_str(), snps_only ? 1 : 0, nullptr, const_counts, &n));
        return n;
    }

    // (extension) LD of the core alignment by site distance over all shards: n_bins = ceil(max_dist / bin_width) bins
    std::vector<pansim_ld_bin> core_ld(const pansim_ld_params &p, uint64_t *sites_used = nullptr)
    {
        const uint64_t n = p.bin_width ? ((uint64_t)p.max_dist + p.bin_width - 1) / p.bin_width : 0;
        std::vector<pansim_ld_bin> bins(std::max<uint64_t>(n, 1));
        gcheck(pansim_group_core_ld(grp_, &p, bins.data(), sites_used));
        bins.resize(n);
        return bins;
    }

    // (extension) linkage of the accessory genes by class (0-0, 0-1, 1-1); the r^2 histogram [3][r2_bins] goes to
    // *hist and the used genes of each group to genes_used[2] if given. The accessory matrix is replicated, so
    // shard 0 answers.
    std::array<pansim_gene_ld_class, 3> gene_ld(const pansim_gene_ld_params &p, std::vector<uint64_t> *hist = nullptr,
                                                uint64_t *genes_used = nullptr)
    {
        std::array<pansim_gene_ld_class, 3> cls{};
        if (hist) hist->assign(3 * (size_t)(p.r2_bins <= 1024 ? p.r2_bins : 0), 0);
        gcheck(pansim_group_gene_ld(grp_, &p, cls.data(), hist && !hist->empty() ? hist->data() : nullptr, genes_used));
        return cls;
    }

    // (extension) pangenome accumulation curves over n_perms random orders of the rows drawn from seed, each
    // [n_perms][N] row-major; the accessory matrix is replicated, so shard 0 answers
    struct GeneAccumulation { std::vector<uint32_t> orders, pan, core, new_genes, unique; };
    GeneAccumulation gene_accumulation(uint64_t seed, uint32_t n_perms)
    {
        GeneAccumulation r;
        const size_t n = n_perms <= PANSIM_GENE_ACC_MAX_PERMS ? (size_t)n_perms * cfg_.pop_size : 0;
        for (auto *v : {&r.orders, &r.pan, &r.core, &r.new_genes, &r.unique}) v->assign(n, 0);
        gcheck(pansim_group_gene_accumulation(grp_, seed, n_perms, r.orders.data(), r.pan.data(), r.core.data(),
                                              r.new_genes.data(), r.unique.data()));
        return r;
    }
    // (extension) the gene frequency spectrum [N + 1]: genes carried by k rows, core_genes in bin N
    std::vector<uint64_t> gene_spectrum()
    {
        std::vector<uint64_t> s((size_t)cfg_.pop_size + 1);
        gcheck(pansim_group_gene_spectrum(grp_, s.data()));
        return s;
    }

    // (extension) record the parent vector of every generation from now on, the last `capacity` kept (0: off)
    void enable_genealogy(uint32_t capacity) { gcheck(pansim_group_enable_genealogy(grp_, capacity)); }
    // (extension) the clonal genealogy of the present population: the node table, and its summary if info is non-null
    std::vector<pansim_genealogy_node> genealogy(pansim_genealogy_info *info = nullptr)
    {
        std::vector<pansim_genealogy_node> nodes(2 * (size_t)cfg_.pop_size);
        pansim_genealogy_info i;
        gcheck(pansim_group_genealogy(grp_, nodes.data(), &i));
        nodes.resize(i.n_nodes);
        if (info) *info = i;
        return nodes;
    }
    // (extension) TMRCA of each pair (range1[k], range2[k]), in generations
    std::vector<uint32_t> tmrca(const std::vector<uint32_t> &range1, const std::vector<uint32_t> &range2)
    {
        std::vector<uint32_t> out(range1.size());
        gcheck(pansim_group_genealogy_tmrca(grp_, range1.data(), range2.data(), range1.size(), out.data()));
        return out;
    }
    // (extension) parsimony changes of the core sites / accessory genes on a node table given as its parent column
    // (pansim_group_core_parsimony / pansim_group_gene_parsimony)
    struct CoreParsimony { pansim_parsimony summary; std::vector<uint32_t> site_changes; std::vector<uint64_t> branch_changes; };
    CoreParsimony core_parsimony(const std::vector<uint32_t> &parent)
    {
        CoreParsimony r{};
        r.site_changes.assign(cfg_.core_size, 0);
        r.branch_changes.assign(parent.size(), 0);
        gcheck(pansim_group_core_parsimony(grp_, parent.data(), (uint32_t)parent.size(), &r.summary, r.site_changes.data(),
                                           r.branch_changes.data()));
        return r;
    }
    struct GeneParsimony { pansim_parsimony summary; std::vector<uint32_t> gene_changes; std::vector<uint64_t> gains, losses; };
    GeneParsimony gene_parsimony(const std::vector<uint32_t> &parent)
    {
        GeneParsimony r{};
        r.gene_changes.assign(cfg_.pan_size, 0);
        r.gains.assign(parent.size(), 0);
        r.losses.assign(parent.size(), 0);
        gcheck(pansim_group_gene_parsimony(grp_, parent.data(), (uint32_t)parent.size(), &r.summary, r.gene_changes.data(),
                                           r.gains.data(), r.losses.data()));
        return r;
    }
    // (extension) the neighbour-joining tree of the present rows, metric 0 core / 1 acc (pansim_group_nj_tree)
    struct NJTree { std::vector<uint32_t> parent; std::vector<double> length; };
    NJTree nj_tree(int metric)
    {
        const uint32_t n = cfg_.pop_size, nodes = n >= 3 ? 2 * n - 2 : n == 2 ? 3 : 1;
        NJTree t{std::vector<uint32_t>(nodes), std::vector<double>(nodes)};
        gcheck(pansim_group_nj_tree(grp_, metric, t.parent.data(), t.length.data()));
        return t;
    }
    // (extension) the Newick text of a node table with branch lengths (pansim_tree_newick)
    std::string tree_newick(const std::vector<uint32_t> &parent, const std::vector<double> &length)
    {
        size_t len = 0;
        check_table(pansim_tree_newick(parent.data(), length.data(), (uint32_t)parent.size(), cfg_.pop_size, nullptr, 0, &len));
        std::string s(len + 1, '\0');
        check_table(pansim_tree_newick(parent.data(), length.data(), (uint32_t)parent.size(), cfg_.pop_size, &s[0], s.size(), &len));
        s.resize(len);
        return s;
    }
    // (extension) {splits of a, splits of b, shared} of two node tables over the rows (pansim_tree_compare_splits)
    std::array<uint64_t, 3> compare_splits(const std::vector<uint32_t> &a, const std::vector<uint32_t> &b)
    {
        std::array<uint64_t, 3> out{};
        check_table(pansim_tree_compare_splits(a.data(), (uint32_t)a.size(), b.data(), (uint32_t)b.size(), cfg_.pop_size, out.data()));
        return out;
    }
    // (extension) the canonical Newick text of a node table (pansim_genealogy_newick)
    std::string newick(const std::vector<pansim_genealogy_node> &nodes)
    {
        size_t len = 0;
        check_newick(pansim_genealogy_newick(nodes.data(), (uint32_t)nodes.size(), cfg_.pop_size, nullptr, 0, &len));
        std::string s(len + 1, '\0');
        check_newick(pansim_genealogy_newick(nodes.data(), (uint32_t)nodes.size(), cfg_.pop_size, &s[0], s.size(), &len));
        s.resize(len);
        return s;
    }

    pansim_ctx *raw() { return ctx_; }          // shard 0 (the whole run when n_gpus() == 1)
    pansim_group *group() { return grp_; }
    const pansim_config &config() const { return cfg_; }

private:
    void check(int rc)
    {
        if (rc != PANSIM_OK) throw Error(rc, pansim_last_error(ctx_));
    }
    void gcheck(int rc)
    {
        if (rc != PANSIM_OK) throw Error(rc, pansim_group_last_error(grp_));
    }
    void check_table(int rc)
    {
        if (rc != PANSIM_OK) throw Error(rc, "the node table breaks the rules of include/pansim_b200.h (section 17 tables)");
    }
    void check_newick(int rc)
    {
        if (rc != PANSIM_OK) throw Error(rc, "pansim_genealogy_newick: the node table is not a tree of that shape");
    }
    // host-driven operators work on one context; a sharded run uses the device-resident calls
    void single(const char *what)
    {
        if (n_gpus() != 1) throw Error(PANSIM_ERR_STATE, std::string(what) + " is a single-GPU call; use step() / run_generations() with --gpus > 1");
    }
    pansim_config cfg_;
    pansim_group *grp_ = nullptr;
    pansim_ctx *ctx_ = nullptr;
};

}  // namespace pansim
