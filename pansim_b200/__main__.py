"""`python -m pansim_b200 [flags]` -- the `pansim` command line (main.rs:17-186).

Same long flags (underscores, capitalised --HR_rate / --HGT_rate), same defaults,
same parsing quirks: pop_size/core_size/pan_genes/core_genes/n_gen are parsed as
f64 and rounded (main.rs:155-167) so `--pop_size 1e3` works; max_distances,
threads and seed are parsed as integers (main.rs:169, 177, 180). --threads is
accepted and ignored (the work runs on the GPU). Extra flags: --device, --all_pairs, --print_diversity, --print_vcf,
--print_ld, --ld_max_dist, --ld_bin_width, --ld_min_minor, --print_genealogy, --print_fasta, --print_snp_alignment,
--print_gene_ld, --gene_ld_bins, --gene_ld_min_minor, --print_gene_accumulation, --gene_accumulation_perms,
--print_parsimony, --print_nj.
"""
from __future__ import annotations

import argparse
import sys

from .params import Params, rust_round
from .simulate import run


def _f64_rounded(s: str) -> int:
    return int(rust_round(float(s)))


def build_parser() -> argparse.ArgumentParser:
    ap = argparse.ArgumentParser(
        prog="pansim",
        description="Runs Wright-Fisher simulation, simulating neutral core genome evolution and "
                    "two-speed accessory genome evolution.", allow_abbrev=False)
    d = Params()
    ap.add_argument("--pop_size", type=_f64_rounded, default=d.pop_size, help="Number of individuals in population.")
    ap.add_argument("--core_size", type=_f64_rounded, default=d.core_size, help="Number of nucleotides in core genome.")
    ap.add_argument("--pan_genes", type=_f64_rounded, default=d.pan_genes,
                    help="Total number of genes in pangenome (core + accessory).")
    ap.add_argument("--core_genes", type=_f64_rounded, default=d.core_genes, help="Number of core genes in pangenome.")
    ap.add_argument("--avg_gene_freq", type=float, default=d.avg_gene_freq)
    ap.add_argument("--n_gen", type=_f64_rounded, default=d.n_gen, help="Number of generations to simulate.")
    ap.add_argument("--max_distances", type=int, default=d.max_distances)
    ap.add_argument("--core_mu", type=float, default=d.core_mu)
    ap.add_argument("--HR_rate", type=float, default=d.HR_rate)
    ap.add_argument("--HGT_rate", type=float, default=d.HGT_rate)
    ap.add_argument("--rate_genes1", type=float, default=d.rate_genes1)
    ap.add_argument("--rate_genes2", type=float, default=d.rate_genes2)
    ap.add_argument("--prop_genes2", type=float, default=d.prop_genes2)
    ap.add_argument("--prop_positive", type=float, default=d.prop_positive)
    ap.add_argument("--pos_lambda", type=float, default=d.pos_lambda)
    ap.add_argument("--neg_lambda", type=float, default=d.neg_lambda)
    ap.add_argument("--seed", type=int, default=d.seed)
    ap.add_argument("--outpref", default=d.outpref, help="Output prefix path.")
    ap.add_argument("--print_dist", action="store_true")
    ap.add_argument("--print_matrices", action="store_true")
    ap.add_argument("--print_selection", action="store_true")
    ap.add_argument("--threads", type=int, default=1, help="Accepted for compatibility; ignored.")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--no_control_genome_size", action="store_true")
    ap.add_argument("--genome_size_penalty", type=float, default=d.genome_size_penalty)
    ap.add_argument("--competition_strength", type=float, default=d.competition_strength)
    ap.add_argument("--device", type=int, default=0, help="(extension) CUDA device ordinal")
    ap.add_argument("--all_pairs", action="store_true",
                    help="(extension) <outpref>.tsv holds every pair i < j in (i, j) order instead of max_distances sampled pairs")
    ap.add_argument("--print_diversity", action="store_true",
                    help="(extension) <outpref>_diversity.tsv: segregating sites, multiallelic sites, pi, Watterson's theta "
                         "and Tajima's D of the core genome every generation; <outpref>_core_sfs.txt: the site frequency "
                         "spectrum of the last generation")
    ap.add_argument("--print_vcf", action="store_true",
                    help="(extension) <outpref>_core_genome.vcf: the core alignment of the last generation as VCF, one "
                         "line per site that differs from the initial row, haploid genotypes against it")
    ap.add_argument("--print_ld", action="store_true",
                    help="(extension) <outpref>_core_ld.tsv: linkage disequilibrium of the core genome of the last generation, "
                         "one line per distance bin: dist_lo, dist_hi, site pairs, pairs with four gametes, mean r^2")
    ap.add_argument("--ld_max_dist", type=int, default=10000, help="(extension) largest site distance of --print_ld")
    ap.add_argument("--ld_bin_width", type=int, default=100, help="(extension) distances per bin of --print_ld")
    ap.add_argument("--ld_min_minor", type=int, default=1,
                    help="(extension) --print_ld uses sites where at least this many rows are derived and at least this many are not")
    ap.add_argument("--print_genealogy", action="store_true",
                    help="(extension) record the parents of every generation; <outpref>_genealogy.nwk: the clonal genealogy of "
                         "the last generation as Newick (leaves ind_<i>, branch lengths in generations); <outpref>_tmrca.tsv: "
                         "the TMRCA of the pair on each line of <outpref>.tsv")
    ap.add_argument("--print_fasta", action="store_true",
                    help="(extension) <outpref>_core_genome.fasta: the core alignment of the last generation as FASTA, one "
                         "record ind_<i> per individual, every site")
    ap.add_argument("--print_snp_alignment", action="store_true",
                    help="(extension) <outpref>_core_snps.fasta: the same records with only the sites where two or more "
                         "letters are present; <outpref>_core_snps_fconst.txt: the constant sites by letter, nA,nC,nG,nT "
                         "(IQ-TREE -fconst)")
    ap.add_argument("--print_gene_ld", action="store_true",
                    help="(extension) <outpref>_gene_ld.tsv: linkage of the accessory genes of the last generation, one line "
                         "per class of gene pair (0-0, 0-1, 1-1 by compartment): class, gene pairs, pairs with four gametes, "
                         "associated pairs, dissociated pairs, mean r^2, then the r^2 histogram")
    ap.add_argument("--gene_ld_bins", type=int, default=20, help="(extension) r^2 histogram bins of --print_gene_ld (1..1024)")
    ap.add_argument("--gene_ld_min_minor", type=int, default=1,
                    help="(extension) --print_gene_ld uses genes present in at least this many rows and absent from at least this many")
    ap.add_argument("--print_gene_accumulation", action="store_true",
                    help="(extension) Roary's pangenome summaries of the last generation: <outpref>_number_of_genes_in_pan_genome"
                         ".Rtab, _number_of_conserved_genes.Rtab, _number_of_new_genes.Rtab, _number_of_unique_genes.Rtab (one "
                         "line per random order of the genomes, keyed by --seed); <outpref>_gene_spectrum.txt; "
                         "<outpref>_summary_statistics.txt (core, soft-core, shell, cloud genes)")
    ap.add_argument("--gene_accumulation_perms", type=int, default=100,
                    help="(extension) random orders of --print_gene_accumulation (1..10000)")
    ap.add_argument("--print_parsimony", action="store_true",
                    help="(extension) parsimony changes on the true genealogy of the last generation: <outpref>_parsimony.tsv "
                         "(core and gene summaries with CI and RI), <outpref>_core_site_changes.txt, <outpref>_gene_changes.txt, "
                         "<outpref>_branch_changes.tsv")
    ap.add_argument("--print_nj", action="store_true",
                    help="(extension) neighbour-joining trees of the last generation on the core and accessory distances: "
                         "<outpref>_core_nj.nwk, <outpref>_acc_nj.nwk, and their splits against the true genealogy in "
                         "<outpref>_nj_rf.tsv")
    return ap


def main(argv=None) -> int:
    ns = vars(build_parser().parse_args(argv))
    device = ns.pop("device")
    all_pairs = ns.pop("all_pairs")
    print_diversity = ns.pop("print_diversity")
    print_vcf = ns.pop("print_vcf")
    print_genealogy = ns.pop("print_genealogy")
    print_fasta = ns.pop("print_fasta")
    print_snp_alignment = ns.pop("print_snp_alignment")
    ld = {k: ns.pop(k) for k in ("print_ld", "ld_max_dist", "ld_bin_width", "ld_min_minor")}
    ld.update({k: ns.pop(k) for k in ("print_gene_ld", "gene_ld_bins", "gene_ld_min_minor", "print_gene_accumulation",
                                      "gene_accumulation_perms", "print_parsimony", "print_nj")})
    p = Params(**ns)
    run(p, outpref=p.outpref, device=device, all_pairs=all_pairs, print_diversity=print_diversity, print_vcf=print_vcf,
        print_genealogy=print_genealogy, print_fasta=print_fasta, print_snp_alignment=print_snp_alignment, **ld)
    return 0                       # the reference exits 0 even when validation fails (main.rs:195-247)


if __name__ == "__main__":
    sys.exit(main())
