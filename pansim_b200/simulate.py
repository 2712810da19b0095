"""Host driver: the reference's `main()` (pansim/src/main.rs:15-564) over the C ABI.

Keeps on the host exactly what north_star leaves there: flag handling,
validation, selection-coefficient setup, initial rows, pair sampling and the
six output writers with the reference's text formats. Everything between
main.rs:435 and :528 runs on the GPU through `Pansim`.

Host randomness (selection coefficients, initial rows, pairs) comes from a
numpy generator seeded with --seed; the reference uses rand's StdRng there, whose
stream cannot be reproduced without the crate, so only the distributions match.
"""
from __future__ import annotations

import math
import sys
from dataclasses import dataclass, field

import numpy as np

from .params import Derived, Params, derive, fmt_f64, validate
from .population import Pansim, compare_splits, diversity_stats, pangenome_classes, standard_deviation


def selection_coefficients(p: Params, pan_size: int, rng: np.random.Generator) -> np.ndarray:
    """main.rs:287-319."""
    s = np.zeros(pan_size, np.float64)
    if p.prop_positive >= 0.0:
        for i in range(pan_size):
            weight = rng.random()
            if weight <= p.prop_positive:
                s[i] = rng.exponential(1.0 / p.pos_lambda)
            else:
                v = rng.exponential(1.0 / p.neg_lambda)
                while v > 1.0:                      # main.rs:309-311
                    v = rng.exponential(1.0 / p.neg_lambda)
                s[i] = -1.0 * v
    return s


def initial_rows(p: Params, d: Derived, rng: np.random.Generator):
    """Population::new x2 (population.rs:199-204, 214-219): one row each."""
    core_row = (1 << rng.integers(0, 4, p.core_size)).astype(np.uint8)
    acc_row = (rng.random(d.pan_size) < d.avg_gene_freq_adj).astype(np.uint8)
    return core_row, acc_row


def sample_pairs(p: Params, rng: np.random.Generator):
    """main.rs:413-427: ordered pairs i != j, with replacement, fixed for the run."""
    r1 = rng.integers(0, p.pop_size, p.max_distances).astype(np.uint32)
    if p.pop_size < 2:
        raise ValueError("pop_size must be >= 2 to sample pairs (gen_range(0..pop_size-1) panics)")
    r2 = rng.integers(0, p.pop_size - 1, p.max_distances).astype(np.uint32)
    r2 = (r2 + (r2 >= r1)).astype(np.uint32)
    return r1, r2


@dataclass
class RunResult:
    core_distances: np.ndarray = None
    acc_distances: np.ndarray = None
    gene_freqs: np.ndarray = None            # accessory genes then core_genes ones (population.rs:857-860)
    per_gen: list = field(default_factory=list)   # (avg_core, std_core, avg_acc, std_acc)
    diversity: list = field(default_factory=list) # per generation: Diversity (--print_diversity)
    sfs: np.ndarray = None                        # SFS of the last generation (--print_diversity)
    ld: object = None                             # CoreLD of the last generation (--print_ld)
    gene_ld: object = None                        # GeneLD of the last generation (--print_gene_ld)
    gene_accumulation: object = None              # GeneAccumulation of the last generation (--print_gene_accumulation)
    gene_spectrum: np.ndarray = None              # gene frequency spectrum of the last generation (--print_gene_accumulation)
    genealogy: object = None                      # Genealogy of the last generation (--print_genealogy)
    core_parsimony: object = None                 # CoreParsimony on the genealogy (--print_parsimony)
    gene_parsimony: object = None                 # GeneParsimony on the genealogy (--print_parsimony)
    nj: dict = None                               # {"core", "acc"}: NJTree of the last generation (--print_nj)
    nj_splits: dict = None                        # {"core", "acc"}: SplitComparison with the genealogy (--print_nj)
    tmrca: np.ndarray = None                      # TMRCA of the sampled pairs (--print_genealogy without --all_pairs)
    selection: np.ndarray = None
    stdout: list = field(default_factory=list)


def run(p: Params, outpref: str | None = None, device: int = 0, out=None, all_pairs: bool = False,
        print_diversity: bool = False, print_vcf: bool = False, print_ld: bool = False, ld_max_dist: int = 10000,
        ld_bin_width: int = 100, ld_min_minor: int = 1, print_genealogy: bool = False, print_fasta: bool = False,
        print_snp_alignment: bool = False, print_gene_ld: bool = False, gene_ld_bins: int = 20,
        gene_ld_min_minor: int = 1, print_gene_accumulation: bool = False,
        gene_accumulation_perms: int = 100, print_parsimony: bool = False, print_nj: bool = False) -> RunResult | None:
    """main.rs:15-564. Returns None where the reference prints a validation message and exits 0.
    all_pairs (extension, BASELINE config 5): `<outpref>.tsv` holds the distances of every pair i < j
    in (i, j) order instead of the max_distances sampled pairs; res.core/acc_distances stay None.
    print_diversity (extension): core-genome diversity every generation, written to
    `<outpref>_diversity.tsv` (segregating, multiallelic, pi, theta_W, Tajima's D) and the site frequency
    spectrum of the last generation to `<outpref>_core_sfs.txt`.
    print_vcf (extension): the core alignment of the last generation as `<outpref>_core_genome.vcf`, written
    after the other outputs (Pansim.write_core_vcf).
    print_ld (extension): linkage disequilibrium of the core alignment of the last generation as
    `<outpref>_core_ld.tsv`, written after the other outputs (Pansim.core_ld with ld_max_dist, ld_bin_width,
    ld_min_minor; write_core_ld).
    print_genealogy (extension): the parents of every generation are recorded on the device from generation 0;
    after the other outputs the genealogy of the last generation goes to `<outpref>_genealogy.nwk` and the TMRCA of
    the pair on each line of `<outpref>.tsv` to `<outpref>_tmrca.tsv` (write_genealogy).
    print_fasta / print_snp_alignment (extension): after the other outputs, the core alignment of the last generation
    as `<outpref>_core_genome.fasta` (every site) / `<outpref>_core_snps.fasta` (the sites where two or more letters
    are present) with `<outpref>_core_snps_fconst.txt`, the constant sites by letter as `nA,nC,nG,nT`
    (Pansim.write_core_fasta).
    print_gene_ld (extension): linkage of the accessory genes of the last generation as `<outpref>_gene_ld.tsv`,
    written after every other output (Pansim.gene_ld with gene_ld_bins, gene_ld_min_minor; write_gene_ld).
    print_gene_accumulation (extension): after every other output, Roary's pangenome summaries of the last generation:
    the accumulation curves over gene_accumulation_perms random orders keyed by p.seed, the gene frequency spectrum
    and the core / soft-core / shell / cloud counts (Pansim.gene_accumulation, Pansim.gene_spectrum;
    write_gene_accumulation).
    print_parsimony (extension): the parents are recorded from generation 0 as for print_genealogy (without its files
    unless that is also given); after every other output, the parsimony changes of the core sites and the accessory
    genes on the genealogy of the last generation (Pansim.core_parsimony, Pansim.gene_parsimony; write_parsimony).
    print_nj (extension): the parents are recorded as for print_parsimony; after every other output, the
    neighbour-joining trees of the last generation on the core and the accessory distances, and their splits against
    the genealogy (Pansim.nj_tree, compare_splits; write_nj)."""
    out = out or sys.stdout
    msgs = validate(p)
    if msgs:
        for m in msgs:
            print(m, file=out)
        return None
    d = derive(p)
    res = RunResult()
    if p.verbose:
        line = f"avg_gene_freq adjusted to {fmt_f64(d.avg_gene_freq_adj)}"      # main.rs:269-271
        print(line, file=out)
        res.stdout.append(line)
    rng = np.random.default_rng(p.seed)                                         # main.rs:289
    sel = selection_coefficients(p, d.pan_size, rng)
    res.selection = sel
    if p.print_selection and outpref:                                            # main.rs:321-331
        with open(outpref + "_selection.tsv", "w") as f:
            f.write("\n".join(fmt_f64(float(x)) for x in sel) + "\n")
    core_row, acc_row = initial_rows(p, d, rng)
    r1, r2 = sample_pairs(p, rng)

    with Pansim.from_params(p, device=device) as sim:
        sim.set_initial(core_row, acc_row)
        sim.set_selection(sel)
        if print_genealogy or print_parsimony or print_nj:
            sim.enable_genealogy(p.n_gen)                                        # after set_initial, which clears the record
        def last_generation_outputs():                                           # main.rs:467-499
            if not all_pairs:
                res.core_distances, res.acc_distances = sim.pairwise_distances(r1, r2)
            res.gene_freqs = sim.gene_frequencies()
            if outpref:
                with open(outpref + ".tsv", "w") as f:
                    if all_pairs:
                        for _, _, cd_, it_, un_ in sim.iter_all_pairs(with_indices=False):
                            c_, a_ = sim.distances_from_counts(cd_, it_, un_)
                            f.write("".join(f"{fmt_f64(float(c))}\t{fmt_f64(float(a))}\n" for c, a in zip(c_, a_)))
                    else:
                        f.write("".join(f"{fmt_f64(float(c))}\t{fmt_f64(float(a))}\n"
                                        for c, a in zip(res.core_distances, res.acc_distances)))
                with open(outpref + "_freqs.txt", "w") as f:
                    f.write("".join(fmt_f64(float(x)) + "\n" for x in res.gene_freqs))

        # Nothing has to come back between generations unless --verbose asks for it: the whole run is one
        # device-resident batch (same states, tests/test_gpu_parity.py). With --print_dist the batch also
        # makes the distance pass and its mean / standard deviation every generation on the device
        # (pansim_run_generations_stats: sums in the reference's left-to-right order, population.rs:87-94).
        device_loop = not p.verbose and not (p.print_dist and all_pairs)
        first_host_gen = 0
        if device_loop:
            if print_diversity:        # one batch: the reduction (and the --print_dist pass) after every generation
                res.diversity, st = sim.run_generations_diversity(0, p.n_gen, *((r1, r2) if p.print_dist else ()))
                if p.print_dist:
                    res.per_gen = [tuple(float(x) for x in row) for row in st]
            elif p.print_dist:
                res.per_gen = [tuple(float(x) for x in row) for row in sim.run_generations_stats(0, p.n_gen, r1, r2)]
            else:
                sim.run_generations(0, p.n_gen)
            first_host_gen = p.n_gen
            last_generation_outputs()
        for j in range(first_host_gen, p.n_gen):                                 # main.rs:429
            sim.step(j)                                                          # main.rs:435-464
            if print_diversity:
                res.diversity.append(sim.core_diversity())
            if j == p.n_gen - 1:
                last_generation_outputs()
            if p.print_dist:                                                     # main.rs:502-519
                # the reference recomputes both passes here even on the last generation;
                # the result is identical, so the last one is reused
                if j == p.n_gen - 1 and not all_pairs:
                    cd, ad = res.core_distances, res.acc_distances
                else:
                    cd, ad = sim.pairwise_distances(r1, r2)
                std_core, avg_core = standard_deviation(cd)
                std_acc, avg_acc = standard_deviation(ad)
                res.per_gen.append((avg_core, std_core, avg_acc, std_acc))
            if p.verbose:                                                        # main.rs:522-526
                l1 = f"Finished gen: {j + 1}"
                l2 = f"avg_gene_freq: {fmt_f64(sim.calc_gene_freq())}"
                print(l1, file=out)
                print(l2, file=out)
                res.stdout += [l1, l2]
        if p.print_dist and outpref:                                             # main.rs:531-548
            with open(outpref + "_per_gen.tsv", "w") as f:
                for avg_core, std_core, avg_acc, std_acc in res.per_gen:
                    f.write(f"{fmt_f64(avg_core)}\t{fmt_f64(std_core)}\t{fmt_f64(avg_acc)}\t{fmt_f64(std_acc)}\n")
        if print_diversity:
            _, res.sfs = sim.core_diversity(sfs=True)
            if outpref:
                write_diversity(outpref, res.diversity, res.sfs, p.pop_size)
        if p.print_matrices and outpref:                                         # main.rs:550-553
            sim.write(outpref)
        if print_vcf and outpref:
            sim.write_core_vcf(outpref + "_core_genome.vcf")
        if print_ld:
            res.ld = sim.core_ld(ld_max_dist, ld_bin_width, ld_min_minor)
            if outpref:
                write_core_ld(outpref, res.ld)
        if print_genealogy:
            res.genealogy = sim.genealogy()
            if not all_pairs:
                res.tmrca = sim.tmrca(r1, r2)
            if outpref:
                write_genealogy(outpref, sim, res.genealogy, None if all_pairs else res.tmrca)
        if print_fasta and outpref:
            sim.write_core_fasta(outpref + "_core_genome.fasta")
        if print_snp_alignment and outpref:
            consts = sim.write_core_fasta(outpref + "_core_snps.fasta", snps_only=True).const_counts
            with open(outpref + "_core_snps_fconst.txt", "w") as f:
                f.write(",".join(str(int(x)) for x in consts) + "\n")
        if print_gene_ld:
            res.gene_ld = sim.gene_ld(gene_ld_bins, gene_ld_min_minor)
            if outpref:
                write_gene_ld(outpref, res.gene_ld)
        if print_gene_accumulation:
            res.gene_accumulation = sim.gene_accumulation(gene_accumulation_perms, p.seed)
            res.gene_spectrum = sim.gene_spectrum()
            if outpref:
                write_gene_accumulation(outpref, res.gene_accumulation, res.gene_spectrum)
        if print_parsimony:
            g = res.genealogy if res.genealogy is not None else sim.genealogy()
            res.core_parsimony = sim.core_parsimony(g)
            res.gene_parsimony = sim.gene_parsimony(g)
            if outpref:
                write_parsimony(outpref, g, res.core_parsimony, res.gene_parsimony)
        if print_nj:
            g = res.genealogy if res.genealogy is not None else sim.genealogy()
            res.nj = {m: sim.nj_tree(m) for m in ("core", "acc")}
            res.nj_splits = {m: compare_splits(t, g, p.pop_size) for m, t in res.nj.items()}
            if outpref:
                write_nj(outpref, res.nj, res.nj_splits)
    return res


def write_nj(outpref: str, trees, splits):
    """`<outpref>_core_nj.nwk` and `<outpref>_acc_nj.nwk`: the neighbour-joining trees (pansim_tree_newick);
    `<outpref>_nj_rf.tsv`: two lines, `core` then `acc`, each NJ splits, genealogy splits, shared, Robinson-Foulds and
    RF / (NJ splits + genealogy splits) (NaN if both are 0), no header."""
    for m in ("core", "acc"):
        with open(f"{outpref}_{m}_nj.nwk", "w") as f:
            f.write(trees[m].newick())
    with open(outpref + "_nj_rf.tsv", "w") as f:
        for m in ("core", "acc"):
            s = splits[m]
            total = s.splits_a + s.splits_b
            f.write(f"{m}\t{s.splits_a}\t{s.splits_b}\t{s.shared}\t{s.rf}\t{fmt_f64(s.rf / total if total else math.nan)}\n")


def clades(parent, n_leaves: int) -> tuple[np.ndarray, np.ndarray]:
    """(first leaf, leaves below) of every node of a node table whose parents have larger ids. Every internal node
    has at least two children, so the pair identifies a clade: the key that joins a per-branch table to a Newick text
    whose internal nodes carry no label."""
    parent = np.asarray(parent, np.int64)
    n = len(parent)
    first = np.full(n, n_leaves, np.int64)
    below = np.zeros(n, np.int64)
    first[:n_leaves] = np.arange(n_leaves)
    below[:n_leaves] = 1
    for k in range(n - 1):
        q = parent[k]
        first[q] = min(first[q], first[k])
        below[q] += below[k]
    return first, below


def write_parsimony(outpref: str, genealogy, core, genes):
    """`<outpref>_parsimony.tsv`: two lines, `core` then `genes`, each characters, variable, tree length, min changes,
    max changes, homoplastic, CI, RI (no header; NaN for an empty denominator); `<outpref>_core_site_changes.txt`: the
    score of each core site in position order; `<outpref>_gene_changes.txt`: the score of each matrix gene in
    `_pangenome.csv` column order; `<outpref>_branch_changes.tsv`: per non-root node in id order, no header: node,
    parent, first leaf, leaves below, branch length (generations), core changes, gene gains, gene losses."""
    with open(outpref + "_parsimony.tsv", "w") as f:
        for name, r in (("core", core), ("genes", genes)):
            f.write("\t".join([name] + [str(int(x)) for x in r[:6]] + [fmt_f64(r.ci), fmt_f64(r.ri)]) + "\n")
    with open(outpref + "_core_site_changes.txt", "w") as f:
        f.write("".join(f"{x}\n" for x in core.site_changes.tolist()))
    with open(outpref + "_gene_changes.txt", "w") as f:
        f.write("".join(f"{x}\n" for x in genes.gene_changes.tolist()))
    parent, time = genealogy.parent, genealogy.time
    first, below = clades(parent, genealogy.n_leaves)
    with open(outpref + "_branch_changes.tsv", "w") as f:
        f.write("".join(f"{k}\t{parent[k]}\t{first[k]}\t{below[k]}\t{time[parent[k]] - time[k]}\t{core.branch_changes[k]}\t"
                        f"{genes.gains[k]}\t{genes.losses[k]}\n" for k in range(len(parent) - 1)))


ROARY_CLASSES = ("Core genes\t(99% <= strains <= 100%)", "Soft core genes\t(95% <= strains < 99%)",
                 "Shell genes\t(15% <= strains < 95%)", "Cloud genes\t(0% <= strains < 15%)",
                 "Total genes\t(0% <= strains <= 100%)")


def write_gene_accumulation(outpref: str, acc, spectrum):
    """Roary's pangenome files: `<outpref>_number_of_genes_in_pan_genome.Rtab`, `_number_of_conserved_genes.Rtab`,
    `_number_of_new_genes.Rtab` and `_number_of_unique_genes.Rtab` (one line per order, N tab-separated counts for
    k = 1..N, no header); `<outpref>_gene_spectrum.txt` (N + 1 lines, genes carried by k rows); and
    `<outpref>_summary_statistics.txt` (core, soft-core, shell, cloud and total genes, Roary's layout)."""
    for name, curve in (("genes_in_pan_genome", acc.pan), ("conserved_genes", acc.core), ("new_genes", acc.new),
                        ("unique_genes", acc.unique)):
        with open(f"{outpref}_number_of_{name}.Rtab", "w") as f:
            f.write("".join("\t".join(map(str, row.tolist())) + "\n" for row in curve))
    with open(outpref + "_gene_spectrum.txt", "w") as f:
        f.write("".join(f"{int(x)}\n" for x in spectrum))
    classes = pangenome_classes(spectrum, len(spectrum) - 1)
    with open(outpref + "_summary_statistics.txt", "w") as f:
        f.write("".join(f"{label}\t{n}\n" for label, n in zip(ROARY_CLASSES, classes)))


def write_gene_ld(outpref: str, gl):
    """`<outpref>_gene_ld.tsv`: one line per class of gene pair, 0-0, 0-1, 1-1 (no header): class, pairs, four-gamete
    pairs, associated, dissociated, mean r^2 (NaN for an empty class), then the r^2 histogram counts."""
    with open(outpref + "_gene_ld.tsv", "w") as f:
        for k, label in enumerate(gl.classes):
            f.write("\t".join([label, str(int(gl.pairs[k])), str(int(gl.four_gamete[k])), str(int(gl.associated[k])),
                               str(int(gl.dissociated[k])), fmt_f64(float(gl.mean_r2[k])), *(str(int(x)) for x in gl.hist[k])]) + "\n")


def write_genealogy(outpref: str, sim, genealogy, tmrca):
    """`<outpref>_genealogy.nwk`: the Newick text; `<outpref>_tmrca.tsv`: one integer per line, the TMRCA of the
    pair on the same line of `<outpref>.tsv` (tmrca = None: every pair i < j in (i, j) order, by row blocks)."""
    with open(outpref + "_genealogy.nwk", "w") as f:
        f.write(genealogy.newick())
    with open(outpref + "_tmrca.tsv", "w") as f:
        if tmrca is not None:
            f.write("".join(f"{int(x)}\n" for x in tmrca))
            return
        N = sim.N
        for i0, i1 in sim.row_blocks():
            ii = np.repeat(np.arange(i0, i1, dtype=np.uint32), [N - 1 - i for i in range(i0, i1)])
            jj = np.concatenate([np.arange(i + 1, N, dtype=np.uint32) for i in range(i0, i1)])
            f.write("".join(f"{int(x)}\n" for x in sim.tmrca(ii, jj)))


def write_core_ld(outpref: str, ld):
    """`<outpref>_core_ld.tsv`: one line per distance bin (no header): dist_lo, dist_hi, pairs, four-gamete pairs,
    mean r^2 (NaN for an empty bin)."""
    with open(outpref + "_core_ld.tsv", "w") as f:
        for lo, hi, n, fg, r2 in zip(ld.dist_lo, ld.dist_hi, ld.pairs, ld.four_gamete, ld.mean_r2):
            f.write(f"{int(lo)}\t{int(hi)}\t{int(n)}\t{int(fg)}\t{fmt_f64(float(r2))}\n")


def write_diversity(outpref: str, diversity, sfs, pop_size: int):
    """`<outpref>_diversity.tsv`: per generation segregating, multiallelic, pi, theta_W, Tajima's D (no header,
    like _per_gen.tsv); `<outpref>_core_sfs.txt`: the N + 1 SFS bins, one per line."""
    with open(outpref + "_diversity.tsv", "w") as f:
        for d in diversity:
            pi, tw, td = diversity_stats(d, pop_size)
            f.write(f"{d.segregating}\t{d.multiallelic}\t{fmt_f64(pi)}\t{fmt_f64(tw)}\t{fmt_f64(td)}\n")
    with open(outpref + "_core_sfs.txt", "w") as f:
        f.write("".join(f"{int(x)}\n" for x in sfs))


def summarize(core_d, acc_d, gene_freqs, n_acc_genes: int) -> dict:
    """Per-run scalars used by the end-to-end KS tests (mirrors oracle ora_summary)."""
    f = np.asarray(gene_freqs[:n_acc_genes], np.float64)
    return dict(
        mean_core=float(np.mean(core_d)), mean_acc=float(np.mean(acc_d)),
        median_core=float(np.median(core_d)), median_acc=float(np.median(acc_d)),
        std_core=float(np.std(core_d)), std_acc=float(np.std(acc_d)),
        mean_gene_freq=float(f.mean()) if n_acc_genes else 0.0,
        frac_freq_lt_01=float((f < 0.1).mean()) if n_acc_genes else 0.0,
        frac_freq_gt_09=float((f > 0.9).mean()) if n_acc_genes else 0.0,
    )
