/*
 * pansim_b200.h -- C ABI of libpansim_b200.so: the B200 (sm_100a) replacement
 * for Pansim's per-generation Wright-Fisher step and pairwise distance pass.
 *
 * The reference has no plugin/FFI layer: the boundary it exposes is the public
 * Rust API of `pansim::population::Population` as `main.rs` drives it
 * (pansim/src/main.rs:429-528). Each entry point below names the reference
 * interface it replaces (file:line under /root/reference/pansim/src/).
 * One opaque context holds BOTH populations (core alignment + accessory
 * presence/absence), because the reference always moves them together with
 * the same parent vector (main.rs:442-464).
 *
 * Conventions
 *  - every pointer argument is caller-owned HOST memory valid for the call,
 *    except arguments whose name starts with `d_` (CUDA device pointers on the
 *    context's device, used by the multi-GPU host plumbing);
 *  - return value 0 = ok, <0 = error (message: pansim_last_error); nothing
 *    unwinds across the boundary (the reference panics via unwrap());
 *  - a context is single-owner and not thread-safe (all Population methods
 *    are called sequentially from the main thread, main.rs:429-528);
 *  - host byte layouts are the reference's: core = one byte per site, one-hot
 *    {1,2,4,8} = A,C,G,T (population.rs:154-162, 201-204); accessory = one
 *    byte per gene in {0,1} (population.rs:214-219); matrices are C-order
 *    [pop_size x columns] (population.rs:164-178).
 *  - there is NO CPU fallback: every call fails with PANSIM_ERR_CUDA when no
 *    sm_100-class device is usable.
 */
#ifndef PANSIM_B200_H
#define PANSIM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PANSIM_OK              0
#define PANSIM_ERR_INVALID    (-1)   /* bad argument / unsupported parameter        */
#define PANSIM_ERR_CUDA       (-2)   /* CUDA runtime failure or no usable device    */
#define PANSIM_ERR_NOMEM      (-3)
#define PANSIM_ERR_WEIGHTS    (-4)   /* WeightedIndex::new would panic (population.rs:440) */
#define PANSIM_ERR_STATE      (-5)   /* call order (e.g. step before set_initial)   */

/* Column shards must start on a multiple of this many core sites (one 2 KiB
 * region of the 2-bit packed row; the RNG is keyed per region lane, so results
 * do not depend on where the shard boundaries are). */
#define PANSIM_SITE_ALIGN 8192u

typedef struct pansim_ctx pansim_ctx;

/* The numbers main.rs:259-287 and :333-367 derive from the command line; they
 * are the kernel parameters. Fill with pansim_config_init() then override. */
typedef struct {
    uint32_t struct_size;          /* = sizeof(pansim_config)                         */
    int32_t  device;               /* CUDA device ordinal                             */
    uint32_t pop_size;             /* N   (main.rs:155-156)                           */
    uint32_t pan_size;             /* G = pan_genes - core_genes (main.rs:259)        */
    uint64_t core_size;            /* L, whole core alignment (main.rs:157-158)       */
    uint64_t site_begin, site_end; /* column shard [begin,end) of the core held by
                                      this context; 0,0 = whole alignment. begin must
                                      be a multiple of PANSIM_SITE_ALIGN. The accessory
                                      matrix is replicated in every context.          */
    uint32_t core_genes;           /* population.rs:168; added to both Jaccard terms  */
    uint32_t n_compartments;       /* 0..2 (main.rs:341-367)                          */
    uint32_t comp_lo[2], comp_hi[2];/* genes with weight 1.0 in compartment c         */
    double   core_mut_mean;        /* n_core_mutations[0]      (main.rs:275-276)      */
    double   hr_mean;              /* n_recombinations_core[0] (main.rs:279); 0 = off */
    double   acc_mut_mean[2];      /* n_pan_mutations[c]       (main.rs:348, 361)     */
    double   hgt_mean[2];          /* n_recombinations_pan[c]  (main.rs:349-366); 0 = off */
    int32_t  avg_gene_num;         /* main.rs:272                                     */
    int32_t  no_control_genome_size;
    double   genome_size_penalty;
    double   competition_strength;
    uint64_t seed;                 /* Philox key (north_star: counter-based RNG keyed
                                      by seed, generation, individual, site block)    */
} pansim_config;

void pansim_config_init(pansim_config *cfg);

/* ---- lifecycle --------------------------------------------------------- */
/* replaces Population::new x2 (population.rs:181-242) minus the random draws,
 * which the host keeps (pansim_set_initial). */
int  pansim_create(const pansim_config *cfg, pansim_ctx **out);
void pansim_destroy(pansim_ctx *ctx);
/* message of the last failure on ctx (ctx == NULL: last pansim_create failure) */
const char *pansim_last_error(const pansim_ctx *ctx);
/* library build info, e.g. "pansim_b200 0.1 sm_100a" */
const char *pansim_version(void);

/* ---- state in / out ---------------------------------------------------- */
/* population.rs:199-230: all N rows start as one row. core_row_onehot is the
 * WHOLE alignment row [core_size]; the context keeps its [site_begin,site_end)
 * slice. acc_row is [pan_size]. */
int pansim_set_initial(pansim_ctx *ctx, const uint8_t *core_row_onehot, const uint8_t *acc_row);
/* arbitrary state (tests, restarts): core [N x local_sites], acc [N x G] */
int pansim_upload_core(pansim_ctx *ctx, const uint8_t *core_onehot);
int pansim_upload_acc(pansim_ctx *ctx, const uint8_t *acc);
/* population.rs:865-897 `write` consumes exactly these matrices */
int pansim_download_core(pansim_ctx *ctx, uint8_t *core_onehot_out);
int pansim_download_acc(pansim_ctx *ctx, uint8_t *acc_out);
/* `A,C,G,T\n` text rows of _core_genome.csv (population.rs:877-879) expanded on
 * the GPU: out holds rows [row_begin,row_end), each 2*local_sites bytes. */
int pansim_export_core_csv(pansim_ctx *ctx, uint32_t row_begin, uint32_t row_end, char *out);
/* the whole _core_genome.csv (population.rs:865-882) written by the library: text expanded on the GPU,
 * streamed through two pinned host chunks (kernel + copy of chunk k+1 overlap the write of chunk k) */
int pansim_write_core_csv(pansim_ctx *ctx, const char *path, uint64_t *bytes_out);
/* selection coefficients s[G] (main.rs:287-319), used as ln(1 + s_j) */
int pansim_set_selection(pansim_ctx *ctx, const double *s);

/* ---- per-generation operators ------------------------------------------ */
/* Population::average_distance on the accessory population
 * (population.rs:753-784 + get_distance :114-151). Result stays on the device
 * for the next pansim_sample_indices; out[N] may be NULL. */
int pansim_average_distance(pansim_ctx *ctx, double *out);

/* Population::sample_indices (population.rs:270-448). avg_pairwise_dists[N]:
 * host vector as main.rs:435-443 passes it; NULL = use the device copy left by
 * pansim_average_distance, or all 1.0 if competition_strength <= 0
 * (main.rs:435-440). parents_out[N] may be NULL. The N draws come from
 * Philox(seed, gen, individual). */
int pansim_sample_indices(pansim_ctx *ctx, uint32_t gen, const double *avg_pairwise_dists,
                          uint32_t *parents_out);
/* main.rs:435-443 in one call: average_distance when competition_strength > 0 (else all 1.0), then
 * sample_indices; both vectors come back behind a single synchronisation. Either output may be NULL. */
int pansim_select_parents(pansim_ctx *ctx, uint32_t gen, double *avg_pairwise_dists_out, uint32_t *parents_out);
/* the intermediate vectors of population.rs:282-437 for parity checks; any may
 * be NULL. Valid after pansim_sample_indices. */
int pansim_get_weights(pansim_ctx *ctx, double *weights, int32_t *num_genes, double *logfit);

/* main.rs:445-464 with parents supplied by the host: next_generation x2 +
 * mutate_alleles x2 + recombine x2 as ONE fused device pass per population
 * (generate mode: events drawn from Philox keyed by seed/gen/row/site-block).
 * The call returns once `parents` has been consumed and the step is enqueued:
 * the core pass keeps running on the device beside the selection calls of the
 * next generation. Every entry point that reads or writes the core alignment
 * (pair counts, downloads, CSV export, uploads, replay steps, timing) waits for
 * it first, and applies the recombination events the pass defers to the next
 * generation (DESIGN.md section 5), so callers always observe the state of
 * population.rs after recombine(). */
int pansim_step_with_parents(pansim_ctx *ctx, uint32_t gen, const uint32_t *parents);
/* whole generation main.rs:435-464 on the device: competition (if
 * competition_strength > 0) -> fitness -> parents -> fused step. */
int pansim_step(pansim_ctx *ctx, uint32_t gen);
/* n consecutive generations gen0..gen0+n-1 without returning to the host */
int pansim_run_generations(pansim_ctx *ctx, uint32_t gen0, uint32_t n);
/* Population::next_generation alone (population.rs:450-465), both populations */
int pansim_next_generation(pansim_ctx *ctx, const uint32_t *parents);
/* parents of the last step (device -> host) */
int pansim_get_parents(pansim_ctx *ctx, uint32_t *parents_out);

/* Replay mode: apply an explicit event list with the reference's store
 * semantics (bit-exact). Lists are flat and in APPLY ORDER, i.e. the order the
 * reference executes `row[site] = allele` (population.rs:508, 537) and
 * `self.pop[[row_idx, col_idx]] = value` (population.rs:745): later entries
 * overwrite earlier ones. Sites/loci are global core coordinates; a sharded
 * context applies the ones that fall in its slice. */
typedef struct {
    const uint32_t *parents;          /* [N]                                          */
    size_t n_core_mut;                /* population.rs:525-538                        */
    const uint32_t *core_mut_row, *core_mut_site;
    const uint8_t  *core_mut_allele;  /* one-hot {1,2,4,8}                            */
    size_t n_acc_flip;                /* population.rs:501-509                        */
    const uint32_t *acc_flip_row, *acc_flip_gene;
    size_t n_hr;                      /* population.rs:728-748 (core)                 */
    const uint32_t *hr_recipient, *hr_locus;
    const uint8_t  *hr_value;         /* snapshotted donor allele, one-hot            */
    size_t n_hgt;                     /* population.rs:728-748 (accessory), value 1   */
    const uint32_t *hgt_recipient, *hgt_gene;
} pansim_events;
int pansim_step_replay(pansim_ctx *ctx, const pansim_events *ev);

/* ---- distance pass / reductions ---------------------------------------- */
/* Population::pairwise_distances for both populations (population.rs:787-837,
 * distances.rs:22-77). Integers out; the host does the f64 divisions of
 * population.rs:822 and :828-830 so text output is bit-identical:
 *   core_diff[k] = hamming_bitwise_fast(row_i,row_j)/2   (differing sites)
 *   inter[k], uni[k] = jaccard_distance_fast(row_i,row_j)
 * Any output may be NULL. In a sharded context core_diff is the partial count
 * over the context's sites (sum over shards = whole count). */
int pansim_pair_counts(pansim_ctx *ctx, const uint32_t *range1, const uint32_t *range2,
                       size_t n_pairs, uint32_t *core_diff, uint32_t *inter, uint32_t *uni);
/* same, outputs left in caller-provided DEVICE buffers (u32[n_pairs]) for an
 * NCCL all-reduce by the host plumbing; returns after the kernels finished. */
int pansim_pair_counts_device(pansim_ctx *ctx, const uint32_t *range1, const uint32_t *range2,
                              size_t n_pairs, void *d_core_diff, void *d_inter, void *d_uni);
/* Exact all-pairs mode (an extension: the reference only samples max_distances
 * pairs with replacement, main.rs:413-427; BASELINE config 5 asks for all
 * N(N-1)/2). Counts for every pair (i, j) with row_begin <= i < row_end and
 * i < j < N, in (i ascending, j ascending) order; the pair list and its plan are
 * generated on the device. n_pairs_out = sum over i of (N-1-i), at most 2^31-1
 * per call (walk the rows in blocks). Outputs may be NULL. */
int pansim_pair_counts_rows(pansim_ctx *ctx, uint32_t row_begin, uint32_t row_end, uint32_t *core_diff,
                            uint32_t *inter, uint32_t *uni, size_t *n_pairs_out);
/* same, outputs left in caller-provided DEVICE buffers (for the NCCL all-reduce
 * of column-sharded contexts) */
int pansim_pair_counts_rows_device(pansim_ctx *ctx, uint32_t row_begin, uint32_t row_end, void *d_core_diff,
                                   void *d_inter, void *d_uni, size_t *n_pairs_out);
/* The per-generation statistics of --print_dist (main.rs:502-519) computed on the device: the
 * distance pass above followed by standard_deviation (population.rs:87-94) of both distance vectors.
 * out[4] = { avg_core, std_core, avg_acc, std_acc }, the columns of _per_gen.tsv (main.rs:546). The
 * four f64 sums are taken strictly left to right like `iter().sum::<f64>()`, so the values are the
 * reference's bit for bit; 32 bytes leave the device instead of three count vectors. */
int pansim_pair_stats(pansim_ctx *ctx, const uint32_t *range1, const uint32_t *range2, size_t n_pairs, double *out);
/* n generations gen0..gen0+n-1, each followed by that pass and its statistics (the loop of
 * main.rs:429-519 under --print_dist), without returning to the host: stats_out[n][4]. */
int pansim_run_generations_stats(pansim_ctx *ctx, uint32_t gen0, uint32_t n, const uint32_t *range1,
                                 const uint32_t *range2, size_t n_pairs, double *stats_out);
/* the two f64 formulas (population.rs:822, :828-830), exported so every host
 * language forms the distances identically */
double pansim_core_distance(uint32_t core_diff, uint64_t core_size);
double pansim_acc_distance(uint32_t inter, uint32_t uni, uint32_t core_genes);

/* Population::gene_frequencies numerators (population.rs:840-856): counts[G] */
int pansim_gene_counts(pansim_ctx *ctx, uint32_t *counts);

/* ---- core-genome diversity (extension: the reference has no such output) ----
 * One column reduction of the packed core alignment on the device (DESIGN.md section 10). Every call
 * observes the state after recombine(), like the pair calls. On a column shard every field and every SFS
 * bin is the partial over the shard's sites; the sum over the shards is the whole-alignment value. */
typedef struct {
    uint64_t sites;          /* local sites counted (site_end - site_begin)                          */
    uint64_t segregating;    /* >= 2 alleles present                                                  */
    uint64_t multiallelic;   /* >= 3 alleles present                                                  */
    uint64_t pair_diff_sum;  /* sum over sites of sum_{a<b} n_a n_b = sum over pairs i<j of core_diff */
} pansim_diversity;
/* per-site allele counts: counts[local_sites][4] = n_A, n_C, n_G, n_T */
int pansim_core_allele_counts(pansim_ctx *ctx, uint32_t *counts);
/* the summaries above; sfs[N+1] (may be NULL): sfs[k] = number of sites where k individuals carry an allele
 * other than the ancestral one, the ancestral row being the row given to pansim_set_initial (uploads do not
 * change it). Asking for the SFS on a context that never had pansim_set_initial fails with PANSIM_ERR_STATE. */
int pansim_core_diversity(pansim_ctx *ctx, pansim_diversity *out, uint64_t *sfs /* [N+1] or NULL */);
/* n generations, each followed by the reduction on the device; with n_pairs > 0 also the --print_dist
 * pass and its statistics, stats_out[n][4] bit-identical to pansim_run_generations_stats (the pair half
 * needs the whole alignment or a communicator, like pansim_run_generations_stats) */
int pansim_run_generations_diversity(pansim_ctx *ctx, uint32_t gen0, uint32_t n, const uint32_t *range1,
                                     const uint32_t *range2, size_t n_pairs, double *stats_out,
                                     pansim_diversity *div_out /* [n] */);
/* out = { pi, theta_W, Tajima's D } from whole-alignment values; needs no device.
 *   pi = pair_diff_sum / C(N,2)   (mean number of differing sites over all pairs)
 *   theta_W = S / a1, a1 = sum_{i=1}^{N-1} 1/i, a2 = sum 1/i^2 (ascending i), S = segregating
 *   D = (pi - S/a1) / sqrt(e1 S + e2 S (S-1)) with b1, b2, c1, c2, e1, e2 of Tajima (1989)
 * D is NaN when S = 0 or the denominator is 0; all three are NaN when N < 2. With four alleles S counts
 * sites, not mutations: a site with three alleles carries at least two mutations, so `multiallelic` shows
 * how far the infinite-sites assumption behind theta_W and D is violated. */
void pansim_diversity_stats(const pansim_diversity *d, uint32_t pop_size, double out[3]);

/* ---- core-genome VCF (extension: the reference writes the alignment only as _core_genome.csv) ----
 * The alignment as VCF 4.2 text, expanded on the device and streamed to the file through the pinned
 * double-buffered pipeline of pansim_write_core_csv (DESIGN.md section 11). Header (each line ends in \n):
 *   ##fileformat=VCFv4.2 / ##source=pansim_b200 / ##contig=<ID=core,length=core_size> /
 *   ##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype"> /
 *   #CHROM POS ID REF ALT QUAL FILTER INFO FORMAT ind_0 .. ind_{N-1}   (tab-separated; ind_i is row i)
 * Then, in position order, one line per site where some row carries an allele other than the ancestral one:
 *   core POS . REF ALT . . . GT g_0 .. g_{N-1}
 * POS = global site index + 1; REF = the site's letter in the row given to pansim_set_initial (uploads do not
 * change it, as for the SFS); ALT = the other letters with a count above zero, in A,C,G,T order, comma-separated;
 * g_i = 0 for REF, else 1 + the index of row i's letter in ALT (haploid, one digit). A site fixed for another
 * letter is written (ALT of one letter, every g_i = 1); a site where every row carries REF is not. A line is
 * 19 + digits(POS) + 2 |ALT| + 2 N bytes. The state is read after recombine(), like every reader.
 * Without pansim_set_initial the calls fail with PANSIM_ERR_STATE; a failed or short write fails with
 * PANSIM_ERR_INVALID. bytes_out (may be NULL) = bytes written. A column-shard context writes its own lines
 * with global POS: the header-less bodies of the shards, concatenated in shard order, are the whole body. */
int pansim_write_core_vcf(pansim_ctx *ctx, const char *path, int with_header, uint64_t *bytes_out);
/* measurement: the site pass (allele counts, line descriptors, offset scan, chunking) and the expansion of
 * every chunk into device memory, each `repeats` times with no copy to the host; mean device ms of one
 * pass (CUDA events) and the bytes of text (header excluded) */
int pansim_core_vcf_kernel_ms(pansim_ctx *ctx, uint32_t repeats, float *site_ms, float *expand_ms, uint64_t *text_bytes);

/* ---- core-genome FASTA alignment (extension: the reference writes the alignment only as _core_genome.csv) ----
 * The alignment as FASTA text for phylogenetic and clustering tools (IQ-TREE, RAxML-NG, FastTree, Gubbins,
 * snp-dists), expanded on the device and streamed to the file through the pinned double-buffered pipeline of
 * pansim_write_core_csv (DESIGN.md section 14).
 *   Whole mode (snps_only = 0): every site of the alignment is a column, in position order.
 *   SNP mode (snps_only != 0): a column is a site where at least two letters are present among the N rows; the
 *     number of columns equals pansim_diversity.segregating. A site fixed for a non-ancestral letter is not a
 *     column. This is the column selection snp-sites makes on a gap-free alignment; it is not the VCF's rule
 *     (pansim_write_core_vcf writes every site that differs from the ancestral row, fixed ones included).
 *   Constant-site counts: const_counts[4] holds, for the sites that are not columns, the number whose letter is
 *     A, C, G and T (in whole mode all four are 0). const_counts summed plus the number of columns equals the
 *     context's sites; in SNP mode they are what IQ-TREE's -fconst a,c,g,t takes.
 *   Bytes: for each row i = 0 .. N-1 in order, one record: ">ind_<i>\n" (the VCF sample names and the Newick leaf
 *     names of the genealogy), the row's letters of the columns (uppercase ACGT, one line, no wrapping), "\n". A
 *     record is 7 + digits(i) + columns bytes; record i starts at byte i (7 + columns) + sum over j < i of digits(j).
 *     With zero columns each record is ">ind_<i>\n\n".
 * The state is read after recombine(), like every reader. The calls need a state (pansim_set_initial or an upload;
 * otherwise PANSIM_ERR_STATE) but not the ancestral row. A path that cannot be created, or a failed or short write,
 * gives PANSIM_ERR_INVALID. The context keeps working after a refused call. columns_out, const_counts (4 values) and
 * bytes_out may be NULL. */
int pansim_write_core_fasta(pansim_ctx *ctx, const char *path, int snps_only, uint64_t *columns_out, uint64_t *const_counts /* [4] or NULL */, uint64_t *bytes_out);
/* The letters of rows [row_begin, row_end): `columns` bytes per row, rows back to back, no headers or separators;
 * *columns_out = the context's columns. out = NULL: only *columns_out. A range past N -> PANSIM_ERR_INVALID. On a
 * column shard the columns are the shard's own: polymorphism is decided per column, so the shards' letters of a row,
 * concatenated in shard order, are the whole row's letters, and their column and constant-site counts sum. */
int pansim_export_core_fasta_rows(pansim_ctx *ctx, int snps_only, uint32_t row_begin, uint32_t row_end, char *out, uint64_t *columns_out);
/* measurement: the site pass (SNP mode: allele counts, polymorphic sites, scan, column list; whole mode: nothing)
 * and the expansion of every chunk of records into device memory, each `repeats` times after a warm-up, with no
 * copy to the host; mean device ms of one pass (CUDA events) and the bytes of the file */
int pansim_core_fasta_kernel_ms(pansim_ctx *ctx, int snps_only, uint32_t repeats, float *site_ms, float *expand_ms, uint64_t *text_bytes);

/* ---- core-genome linkage disequilibrium (extension: the reference has no two-site statistic) ----
 * r^2 and four-gamete pairs binned by the distance between two sites, the joint counts of the site pairs formed
 * on the tensor cores (DESIGN.md section 12). The state is read after recombine(), like every reader.
 * Let n = N. At a local site a row is DERIVED when its letter differs from the site's letter in the ancestral row
 * (the row given to pansim_set_initial), the convention of the SFS and of VCF GT != 0; multiallelic sites are
 * collapsed to derived / ancestral. a = the derived count of a site; the site is USED when
 * 1 <= min_minor <= min(a, n - a). The pairs are used sites i < j (global 0-based indices) with
 * 1 <= d = j - i <= max_dist; pair (i, j) goes to bin b = (d - 1) / bin_width. There are
 * n_bins = ceil(max_dist / bin_width) bins; bin b covers distances b*w + 1 .. min((b + 1)*w, max_dist).
 * Per pair, with c = the number of rows derived at both sites:
 *   D = n*c - a_i*a_j, exact in int64;
 *   inv_x = 1.0 / (double)(a_x*(n - a_x)), the product exact, the division IEEE round-to-nearest, once per site;
 *   r2 = (((double)D * (double)D) * inv_i) * inv_j, each product rounded on its own (no fused or reordered operation);
 *   q = round-half-even(r2 * 2^32) as uint64;
 *   four gametes iff c > 0, a_i - c > 0, a_j - c > 0 and n - a_i - a_j + c > 0.
 * |D| <= n^2/4 < 2^53, so D, a(n - a) and their conversions to double are exact for every N a context can hold.
 * Per bin the call returns the pairs, the four-gamete pairs and sum q as an exact 128-bit integer (r2_hi, r2_lo).
 * Every output is an integer: neither the grid nor the shard split changes a bit.
 *
 * next: NULL, or the context holding the sites right after ctx's (next.site_begin == ctx.site_end, same N). Without
 * it ctx counts the pairs whose sites both lie in its own range. With it ctx also counts the pairs whose second site
 * lies among next's first max_dist sites, made on next's device and copied over as a halo (cudaMemcpyPeerAsync);
 * pairs with both sites in the halo belong to next. sites_used (may be NULL) counts ctx's own used sites only. So
 * over column shards s = 0..k-1 the sum of pansim_core_ld(shard s, shard s+1) is the single-context result bit for
 * bit; pansim_group_core_ld is that sum. Under a communicator (pansim_comm_init_rank) a rank's call counts only its
 * own pairs: there is no halo exchange between processes.
 * Errors: no pansim_set_initial -> PANSIM_ERR_STATE; max_dist, bin_width or min_minor = 0, a next that is not
 * adjacent or has another N, or max_dist above next's local sites (group: above the narrowest shard) ->
 * PANSIM_ERR_INVALID. The context keeps working after a refused call. The site-major bit rows (one bit per row and
 * used site) are allocated on first use and kept with the context. */
typedef struct { uint32_t max_dist, bin_width, min_minor; } pansim_ld_params;
typedef struct { uint64_t pairs, four_gamete, r2_hi, r2_lo; } pansim_ld_bin;
int pansim_core_ld(pansim_ctx *ctx, pansim_ctx *next, const pansim_ld_params *p,
                   pansim_ld_bin *bins /* [n_bins] */, uint64_t *sites_used);
/* measurement (next = NULL): the site pass (allele counts, used sites, scan, compaction), the transpose to bit rows
 * and the pair pass (tile list and pair kernel), each `repeats` times after one warm-up call; mean device ms of one
 * pass (CUDA events) and the pairs counted */
int pansim_core_ld_kernel_ms(pansim_ctx *ctx, const pansim_ld_params *p, uint32_t repeats,
                             float *site_ms, float *transpose_ms, float *pair_ms, uint64_t *pairs);
/* mean r^2 of a bin, needs no device: (ldexp((double)r2_hi, 32) + ldexp((double)r2_lo, -32)) / (double)pairs in
 * that order, NaN when pairs = 0, so every host prints the same digits */
double pansim_ld_mean_r2(const pansim_ld_bin *b);

/* ---- accessory-gene linkage (extension: the reference writes single-gene frequencies only) ----
 * r^2, associated, dissociated and four-gamete gene pairs by compartment class, the joint presence counts of the
 * gene pairs formed on the tensor cores (DESIGN.md section 15). Presence is absolute, so no ancestral row is needed.
 * Let n = N. Gene g in [0, G) is PRESENT in row r when its bit is set; a_g = the rows carrying g (the numbers
 * pansim_gene_counts returns). group(g) = 1 if n_compartments == 2 and comp_lo[1] <= g < comp_hi[1], else 0 (with
 * both compartments, group 1 is the genes of --rate_genes2, main.rs:341-367). A gene is USED when
 * 1 <= min_minor <= min(a, n - a); genes at or past G are never used. The pairs are all pairs of used genes g < h
 * (there is no window: gene indices carry no position); the class of a pair is group(g) + group(h):
 * 0 = "0-0", 1 = "0-1", 2 = "1-1". Per pair, with c = the rows carrying both genes, exactly as pansim_core_ld:
 *   D = n*c - a_g*a_h, exact in int64;
 *   inv_x = 1.0 / (double)(a_x*(n - a_x)), the product exact, the division IEEE round-to-nearest, once per gene;
 *   r2 = (((double)D * (double)D) * inv_g) * inv_h, each product rounded on its own;
 *   q = round-half-even(r2 * 2^32) as uint64;
 *   four gametes iff c > 0, a_g - c > 0, a_h - c > 0 and n - a_g - a_h + c > 0;
 *   the pair is ASSOCIATED when D > 0 and DISSOCIATED when D < 0;
 *   its r^2 histogram bin is b = min((q * r2_bins) >> 32, r2_bins - 1) in uint64 (q <= 2^32, r2_bins <= 1024).
 * Per class the call returns the pairs, the four-gamete pairs and sum q as an exact 128-bit integer in `ld` (so
 * pansim_ld_mean_r2(&classes[k].ld) is the class mean), and the associated and dissociated pairs;
 * hist[class * r2_bins + b] = the pairs of that class in bin b; genes_used[group] = the used genes of each group.
 * Every output is an integer: neither the grid nor the shard count changes a bit. G = 0 or N < 2 gives all zeros.
 * Errors: no state (pansim_set_initial or pansim_upload_acc) -> PANSIM_ERR_STATE; r2_bins = 0, r2_bins > 1024 or
 * min_minor = 0 -> PANSIM_ERR_INVALID. The context keeps working after a refused call. The gene-major presence bit
 * rows (one bit per row and used gene) are allocated on first use and kept with the context. */
typedef struct { uint32_t r2_bins, min_minor; } pansim_gene_ld_params;
typedef struct { pansim_ld_bin ld; uint64_t associated, dissociated; } pansim_gene_ld_class;
int pansim_gene_ld(pansim_ctx *ctx, const pansim_gene_ld_params *p, pansim_gene_ld_class classes[3],
                   uint64_t *hist /* [3][r2_bins] or NULL */, uint64_t genes_used[2] /* or NULL */);
/* measurement: the gene pass (presence counts, used genes, scan, compaction), the transpose to bit rows and the
 * pair pass (zeroed outputs and pair kernel), each `repeats` times after one warm-up call; mean device ms of one
 * pass (CUDA events) and the pairs counted */
int pansim_gene_ld_kernel_ms(pansim_ctx *ctx, const pansim_gene_ld_params *p, uint32_t repeats,
                             float *gene_ms, float *transpose_ms, float *pair_ms, uint64_t *pairs);

/* ---- pangenome accumulation curves and gene frequency spectrum (extension: the reference writes _freqs.txt) ----
 * Roary's pangenome summaries of the accessory state (DESIGN.md section 16). N = pop_size, G = pan_size (the matrix
 * genes), c0 = cfg.core_genes: the c0 genes are carried by every row and are not in the matrix (_freqs.txt appends
 * them as 1.0, pansim_acc_distance adds them). a_g = the rows carrying matrix gene g (the numbers pansim_gene_counts
 * returns). Bits at or past G in a row's last word are never counted.
 * ORDERS. Order p (0 <= p < P) is a permutation o_p of 0..N-1 drawn by Fisher-Yates: start from the identity; for
 * i = N-1 down to 1 swap o[i] and o[j], j = (uint32)(((uint64)r * (i+1)) >> 32), r = .x of philox4x32_10 (common.cuh)
 * with key = (lo32(seed), hi32(seed)) and counter = {i, p, 0, PANSIM_GENE_ACC_ORDER_TAG}. No simulation stream has
 * that counter word 3 (theirs are (stream << 16) | q below 0x00090000, or 0x01000000 + e for recombination events).
 * The draw touches no simulation stream and changes no state.
 * CURVES. x_k = row o_p[k-1], k = 1..N; per order and k:
 *   pan(k)    = c0 + the matrix genes present in at least one of x_1..x_k;
 *   core(k)   = c0 + the matrix genes present in all of x_1..x_k;
 *   new(k)    = the matrix genes present in x_k and in none of x_1..x_{k-1}, + c0 when k = 1 (pan(k) = sum_{j<=k} new(j));
 *   unique(k) = the matrix genes present in exactly one of x_1..x_k, + c0 when k = 1 (every gene is unique then).
 * Every value is a uint32 (<= G + c0); no output depends on the grid, the chunking or the shard count.
 * SPECTRUM. spectrum[k], k = 0..N = the matrix genes with a_g = k, + c0 in bin N. Bin 0 holds the matrix genes no row
 * carries; they are not in the pangenome.
 * CLASSES (Roary's thresholds as integer tests on a gene carried by a >= 1 rows): core if 100 a >= 99 N, else soft
 * core if 100 a >= 95 N, else shell if 100 a >= 15 N, else cloud; total = the sum of the four. The c0 genes are core.
 * The integer rule is the definition; Roary's floating-point rounding at a boundary is not promised.
 * The state is read like pansim_gene_counts: acc[acc_cur] on the context's stream, so it follows every enqueued step.
 * Errors: no accessory state (pansim_set_initial or pansim_upload_acc) -> PANSIM_ERR_STATE; n_perms = 0 or
 * n_perms > PANSIM_GENE_ACC_MAX_PERMS -> PANSIM_ERR_INVALID. The context keeps working after a refused call. The
 * orders, per-step counts and curves (32 bytes per order and row) are allocated on first use and kept with the context;
 * the orders stay on the device unless `orders` is non-NULL. */
#define PANSIM_GENE_ACC_ORDER_TAG 0x00A00000u
#define PANSIM_GENE_ACC_MAX_PERMS 10000u
/* every output is [n_perms][N] and may be NULL */
int pansim_gene_accumulation(pansim_ctx *ctx, uint64_t seed, uint32_t n_perms, uint32_t *orders, uint32_t *pan,
                             uint32_t *core, uint32_t *new_genes, uint32_t *unique);
/* measurement: the order draw and the accumulation (zeroed counts, chunk summaries, walk, curves), each `repeats`
 * times after one warm-up call; mean device ms of one pass (CUDA events); bytes_read = n_perms * N * ceil(G/32) * 4,
 * the rows as the walk reads them */
int pansim_gene_accumulation_kernel_ms(pansim_ctx *ctx, uint64_t seed, uint32_t n_perms, uint32_t repeats,
                                       float *order_ms, float *accum_ms, uint64_t *bytes_read);
/* spectrum[N + 1] as above (presence counts of acc_gene_counts_kernel, binned on the device) */
int pansim_gene_spectrum(pansim_ctx *ctx, uint64_t *spectrum);
/* out = { core, soft core, shell, cloud, total } of a spectrum[pop_size + 1]; needs no device, so every host prints
 * the same numbers */
void pansim_pangenome_classes(const uint64_t *spectrum, uint32_t pop_size, uint64_t out[5]);

/* ---- clonal genealogy (extension: the reference keeps no pedigree) -------
 * The parent vectors the generations were drawn with, recorded on the device, and the genealogy of the present
 * population traced from them (DESIGN.md section 13). Both populations share it: next_generation gathers the core and
 * the accessory rows by the same vector.
 *
 * Record. Once recording is enabled, each call that advances the population by one generation appends that
 * generation's parent vector H (u32[N], child -> parent index in the previous generation): pansim_step,
 * pansim_run_generations, pansim_run_generations_stats, pansim_run_generations_diversity, pansim_step_with_parents,
 * pansim_next_generation and pansim_step_replay. The record keeps the last `capacity` vectors as a ring. Let T be the
 * number of vectors kept, H_1 .. H_T oldest first. Generation 0 is the population before H_1; generation T is the
 * present. pansim_set_initial, pansim_upload_core, pansim_upload_acc and enabling again clear the record (T = 0).
 *
 * Lineages: a_T(i) = i, a_{t-1}(i) = H_t[a_t(i)].
 * Nodes:
 *   - Leaves are nodes 0 .. N-1. Leaf i is present individual i: time 0, individual = i.
 *   - An internal node is created at generation t for each individual x such that at least two distinct
 *     generation-(t+1) ancestors of present individuals have x as their parent: |{a_{t+1}(i) : a_t(i) = x}| >= 2.
 *     Its time is T - t and its individual is x.
 *   - Internal nodes are numbered N, N+1, ... from the present backwards (time ascending); within one generation
 *     they are ordered by the smallest leaf below them, ascending.
 *   - If more than one lineage remains at generation 0, a virtual root is added last: time T, individual =
 *     0xFFFFFFFF, its children the remaining lineages' top nodes. Otherwise the last merge (the MRCA) is the root,
 *     and the trace stops there even when t > 0.
 *   - The root's parent is 0xFFFFFFFF. There are at most 2N nodes, and every parent has a larger id than its child.
 * TMRCA(i, j) = the time of the lowest common ancestor of leaves i and j: 0 for i = j, T under a virtual root
 * ("not coalesced within the record").
 * Newick: a leaf is `ind_<i>` (the sample names of the VCF); an internal node is `(` its children, `,`-separated,
 * `)` with no label; every non-root node is followed by `:` and its branch length parent.time - time as a decimal
 * integer; children are ordered by the smallest leaf below them, ascending; the text ends with `;` and `\n`. With
 * N = 1 the tree is `ind_0;\n`. This ordering makes the string canonical: the same history gives the same bytes on
 * every host and every shard count. Every output is an integer; no grid, stream or shard split changes a byte.
 *
 * Cost while recording: one device-to-device copy of N x 4 bytes per generation on a stream of its own, ordered after
 * the parent draw by an event; the selection chain, its graphs and the core step are unchanged. With recording off no
 * call, event or graph differs. The trace (one CTA) and the TMRCA walk run when asked for.
 *
 * pansim_enable_genealogy allocates the ring, capacity x N x 4 bytes of device memory (plus 52 N bytes for the trace);
 * a failed allocation returns PANSIM_ERR_NOMEM and leaves recording off. capacity = 0 turns recording off and frees
 * the ring. pansim_genealogy traces on the device and copies back the node table (nodes[2N], may be NULL) and the
 * summary; lineages_at_start = 1 means the MRCA was found. pansim_genealogy_history copies the record itself,
 * out[kept][N] oldest first. pansim_genealogy_tmrca uses the device node table of the current record (traced again
 * if the record changed since the last trace); an index >= N returns PANSIM_ERR_INVALID. Before
 * pansim_enable_genealogy these return PANSIM_ERR_STATE. The context keeps working after a refused call. */
typedef struct { uint32_t parent, individual, time; } pansim_genealogy_node;
typedef struct { uint64_t generations_total; uint32_t generations_kept, n_nodes, lineages_at_start; } pansim_genealogy_info;
int pansim_enable_genealogy(pansim_ctx *ctx, uint32_t capacity);
int pansim_genealogy(pansim_ctx *ctx, pansim_genealogy_node *nodes /* [2N] */, pansim_genealogy_info *info);
int pansim_genealogy_history(pansim_ctx *ctx, uint32_t *out /* [kept][N], oldest first */);
int pansim_genealogy_tmrca(pansim_ctx *ctx, const uint32_t *r1, const uint32_t *r2, size_t n_pairs, uint32_t *tmrca);
/* Newick text of a node table (as pansim_genealogy returns it; n_leaves = N), needs no device. Iterative: any depth.
 * *len = the length of the text, terminating NUL excluded. out = NULL: only *len. Otherwise cap must hold the text
 * and its NUL; if it does not, PANSIM_ERR_INVALID with *len set. A table that is not a tree of that shape (root not
 * last, a parent not above its child, a leaf as parent, a branch of negative length) -> PANSIM_ERR_INVALID. */
int pansim_genealogy_newick(const pansim_genealogy_node *nodes, uint32_t n_nodes, uint32_t n_leaves, char *out,
                            size_t cap, size_t *len);

/* ---- parsimony on the true genealogy (extension) --------------------------
 * How many changes each core site and each accessory gene needs on a rooted tree of the present rows (DESIGN.md
 * section 17): the per-character, per-branch and summary counts of homoplasy tools, on the genealogy the run made.
 * TREE. A node table parent[n_nodes]: leaves are nodes 0 .. N-1, leaf i = row i; every non-root node has a parent with
 * a larger id (ascending ids visit children before parents); the root is the last node, parent 0xFFFFFFFF; every
 * internal node has at least 2 children, so N <= n_nodes <= 2N - 1 (with N = 1 the single leaf is the root).
 * pansim_genealogy's table satisfies this (pass its .parent column); any rooted tree over the rows does once it is
 * renumbered in postorder. A table that breaks a rule -> PANSIM_ERR_INVALID (checked on the host).
 * CHARACTERS. Core: every site of the context's local column range, state = the letter, A < C < G < T. Genes: the G
 * matrix genes, state = absent < present. Padding (the tail of a row's last word, region padding, bits at or past G)
 * never counts.
 * SCORE (Hartigan 1973; Fitch 1971 on binary nodes). A leaf's set is {its state}. An internal node v with children
 * u_1 .. u_k: n_x = |{j : x in S(u_j)}|, m_v = max_x n_x, S(v) = {x : n_x = m_v}, and v contributes k - m_v.
 * score(c) = the sum over internal nodes = the least number of branches whose ends differ at c over all assignments
 * of states to the internal nodes. A node with k >= 3 children is a hard polytomy: each child branch is a branch.
 * SUMMARY. characters; variable = characters with >= 2 states among the leaves; tree_length S = sum of scores;
 * min_changes M = sum (distinct states - 1); max_changes G = sum (N - max_x count_x), the score on a star tree;
 * homoplastic = characters with score > distinct - 1. pansim_parsimony_indices (no device) forms CI = M / S and
 * RI = (G - S) / (G - M), NaN where the denominator is 0, so every host prints the same bytes.
 * RECONSTRUCTION (one optimal assignment, fixed by rule). The root takes the smallest state of S(root); a non-root
 * internal node takes its parent's state if that is in its set, else the smallest state of its set; a leaf takes its
 * own state. branch_changes[v] (core) = the characters whose state at v differs from the state at parent(v);
 * gains[v] / losses[v] (genes) = the characters absent at the parent and present at v / the reverse. Root entries
 * are 0. The rule is optimal (the cost of v's subtree and branch given the parent state y is s_v + [y not in S(v)]),
 * so sum_v branch_changes[v] = S (core) and sum_v gains[v] + losses[v] = S (genes).
 * Every output is an integer: no slab count, grid or shard split changes a bit. The state is read on the context's
 * stream after every enqueued step (pending recombination applied first). Every output pointer may be NULL.
 * Scratch: (n_nodes - N) x 16 bytes per column of 32 sites (core) or x 8 bytes per word of 32 genes, allocated for the
 * call in slabs of columns under a budget (the smaller of 16 GiB and half the free device memory;
 * PANSIM_PARSIMONY_SCRATCH_MB overrides it) and freed before it returns.
 * Errors: no state (pansim_set_initial or pansim_upload_*) -> PANSIM_ERR_STATE; a bad table -> PANSIM_ERR_INVALID;
 * scratch that cannot be allocated -> PANSIM_ERR_NOMEM. The context keeps working after a refused call. */
typedef struct { uint64_t characters, variable, tree_length, min_changes, max_changes, homoplastic; } pansim_parsimony;
int pansim_core_parsimony(pansim_ctx *ctx, const uint32_t *parent, uint32_t n_nodes, pansim_parsimony *out,
                          uint32_t *site_changes /* [local L] */, uint64_t *branch_changes /* [n_nodes] */);
int pansim_gene_parsimony(pansim_ctx *ctx, const uint32_t *parent, uint32_t n_nodes, pansim_parsimony *out,
                          uint32_t *gene_changes /* [G] */, uint64_t *gains /* [n_nodes] */, uint64_t *losses /* [n_nodes] */);
/* measurement: the parsimony kernels of one call (every slab; genes != 0: the gene pass) `repeats` times after one
 * warm-up pass; mean device ms of one pass (CUDA events); bytes_read = columns x (2 N x row bytes of a column + (3 x
 * internal nodes - 1) x set bytes), the rows and scratch as the walk reads them; slabs = the slabs of one pass.
 * Any output may be NULL. */
int pansim_parsimony_kernel_ms(pansim_ctx *ctx, const uint32_t *parent, uint32_t n_nodes, int genes, uint32_t repeats,
                               float *ms, uint64_t *bytes_read, uint32_t *slabs);
/* CI and RI of a summary (either may be NULL); needs no device */
void pansim_parsimony_indices(const pansim_parsimony *p, double *ci, double *ri);

/* ---- neighbour-joining trees from the all-pairs distances (extension) -----
 * The tree PopPUNK or snp-dists -> RapidNJ would infer from the present rows, on the device (DESIGN.md section 18),
 * and an exact split comparison with any other tree over the same leaves (the true genealogy, for instance).
 * DISTANCES. metric 0 (core): d_ij = pansim_core_distance(core_diff, core_size). metric 1 (acc): d_ij =
 * pansim_acc_distance(inter, uni, core_genes), except d = 0 where uni + core_genes = 0. These are the values of
 * <outpref>.tsv over every pair i < j, whatever max_distances is. pansim_nj_tree_matrix takes a caller's matrix as its
 * upper triangle, row-major (d(0,1), d(0,2), .. d(0,n-1), d(1,2), ..); a non-finite or negative entry ->
 * PANSIM_ERR_INVALID. Core on a context with core_size = 0 -> PANSIM_ERR_INVALID; core on a column shard without a
 * communicator -> PANSIM_ERR_STATE (its counts are partial). Under a communicator the counts are summed first
 * (comm_allreduce_counts), so every rank computes the same tree.
 * ALGORITHM (Saitou & Nei 1987, with Studier & Keppler's 1988 Q). IEEE binary64, round-to-nearest, nothing contracted,
 * every operation in the order written here, so a float64 numpy transcription reproduces every bit.
 *  - Active nodes sit in an ordered list of slots, initially leaves 0 .. N-1 in order.
 *  - R_a = sum_b d_ab, summed left to right over ascending b (d_aa = 0), once.
 *  - While k = active > 3: the slots a < b minimising Q_ab = ((k - 2) * d_ab - R_a) - R_b, compared as doubles, ties to
 *    the smaller a, then the smaller b (no grid, tile or reduction order enters).
 *  - delta_a = (d_ab + (R_a - R_b) / (k - 2)) * 0.5, delta_b = d_ab - delta_a (negative lengths are kept, as ape::nj
 *    keeps them).
 *  - Join t (from 0) makes node N + t; it takes slot a, slot b leaves the list, the other slots keep their order.
 *  - Every other active c: d_uc = ((d_ac + d_bc) - d_ab) * 0.5; R_c = ((R_c - d_ac) - d_bc) + d_uc;
 *    R_u = (((R_a - d_ab) + (R_b - d_ab)) - (k - 2) * d_ab) * 0.5.
 *  - The last slots x < y < z become the root 2N - 3, children in that order, delta_x = ((d_xy + d_xz) - d_yz) * 0.5,
 *    delta_y = ((d_xy + d_yz) - d_xz) * 0.5, delta_z = ((d_xz + d_yz) - d_xy) * 0.5.
 *  - N = 2: root 2, both branches d_01 * 0.5. N = 1: the single leaf.
 * OUTPUT. parent[n_nodes] (root 0xFFFFFFFF) and length[n_nodes] (branch above each node, root 0), n_nodes = 2N - 2
 * for N >= 3, 3 for N = 2, 1 for N = 1: a node table in the sense of pansim_core_parsimony (parents above children,
 * root last, every internal node with >= 2 children), so the parsimony calls take it unchanged.
 * The matrix (N x N doubles, padded rows; plus a second buffer for the first compaction) is allocated for the call and
 * freed before it returns: PANSIM_ERR_NOMEM if it cannot be, and the context keeps working. No state
 * (pansim_set_initial or pansim_upload_*) -> PANSIM_ERR_STATE. */
int pansim_nj_tree(pansim_ctx *ctx, int metric /* 0 core, 1 acc */, uint32_t *parent, double *length);
int pansim_nj_tree_matrix(pansim_ctx *ctx, const double *upper /* n (n - 1) / 2 */, uint32_t n, uint32_t *parent,
                          double *length);
/* measurement: one warm-up call, then `repeats` calls; mean device ms of the matrix build (pair counts, scatter, R)
 * and of the join loop (scans, joins, compactions, the last three) by CUDA events; bytes_scanned = sum over the
 * iterations of the stored upper triangle the scan reads x 8 bytes; compactions of one call. Any output may be NULL. */
int pansim_nj_kernel_ms(pansim_ctx *ctx, int metric, uint32_t repeats, float *build_ms, float *join_ms,
                        uint64_t *bytes_scanned, uint32_t *compactions);
/* Newick of a node table with branch lengths (no device): leaves ind_<i>, children ordered by their smallest leaf,
 * lengths "%.17g" (they round-trip), the same writer as pansim_genealogy_newick; out / cap / len as there. A table
 * that breaks the node-table rules -> PANSIM_ERR_INVALID. */
int pansim_tree_newick(const uint32_t *parent, const double *length, uint32_t n_nodes, uint32_t n_leaves, char *out,
                       size_t cap, size_t *len);
/* SPLITS (no device). Every non-root edge of a node table over n_leaves leaves cuts the leaves in two; splits(T) is
 * the set of distinct bipartitions with both sides of >= 2 leaves (trivial splits excluded; the two edges of a binary
 * root give one split). out = {|splits(A)|, |splits(B)|, |shared|}; Robinson-Foulds = out[0] + out[1] - 2 out[2].
 * Exact (leaf sets, not hashes), for polytomies and a virtual root alike. A table that breaks the rules ->
 * PANSIM_ERR_INVALID. */
int pansim_tree_compare_splits(const uint32_t *parent_a, uint32_t n_a, const uint32_t *parent_b, uint32_t n_b,
                               uint32_t n_leaves, uint64_t out[3]);

/* ---- multi-GPU: column shards of one alignment --------------------------
 * (SURVEY.md 8e; the reference is one shared-memory process, population.rs has no analogue.)
 * Every shard context holds all individuals for [site_begin, site_end) and a replica of the
 * accessory matrix; parents, flips and HGT are recomputed identically everywhere from the same
 * counters, so the generation step needs no exchange. The distance pass has one: the per-pair partial
 * core counts are summed over the shards with NCCL inside the library.
 *
 * (a) one process per GPU (torchrun, MPI): rank 0 calls pansim_comm_unique_id, the host plumbing
 *     broadcasts the 128 bytes, every rank calls pansim_comm_init_rank on its context. From then on
 *     pansim_pair_counts / _device / _rows / _rows_device / pansim_pair_stats return WHOLE-alignment
 *     core counts on every rank (ncclAllReduce on the context's stream before the read-back).
 * (b) one process, several GPUs: pansim_group_* below (ncclCommInitAll). */
#define PANSIM_COMM_ID_BYTES 128
int pansim_comm_unique_id(void *id_out);
int pansim_comm_init_rank(pansim_ctx *ctx, int n_ranks, int rank, const void *id);
int pansim_comm_info(pansim_ctx *ctx, int *n_ranks, int *rank);

/* (b) one process, several GPUs. The configuration describes the WHOLE alignment (site_begin =
 *     site_end = 0, `device` ignored); devices == NULL means 0..n_devices-1. Calls mirror the
 *     single-context ones and cite the same reference lines; each enqueues on every shard before it
 *     synchronises, so a single host thread keeps all devices busy. */
typedef struct pansim_group pansim_group;
/* column shard [begin, end) that shard i of n holds (whole 8192-site regions; needs no device) */
int  pansim_shard_bounds(uint64_t core_size, int n_shards, int shard, uint64_t *site_begin, uint64_t *site_end);
int  pansim_group_create(const pansim_config *cfg, int n_devices, const int *devices, pansim_group **out);
void pansim_group_destroy(pansim_group *g);
const char *pansim_group_last_error(const pansim_group *g);   /* g == NULL: last pansim_group_create failure */
int  pansim_group_size(const pansim_group *g);
pansim_ctx *pansim_group_ctx(pansim_group *g, int shard);     /* borrowed; shard i holds sites [begin_i, end_i) */
int pansim_group_set_initial(pansim_group *g, const uint8_t *core_row_onehot, const uint8_t *acc_row);
int pansim_group_set_selection(pansim_group *g, const double *s);
int pansim_group_run_generations(pansim_group *g, uint32_t gen0, uint32_t n);            /* main.rs:435-464 x n */
int pansim_group_pair_counts(pansim_group *g, const uint32_t *range1, const uint32_t *range2, size_t n_pairs,
                             uint32_t *core_diff, uint32_t *inter, uint32_t *uni);      /* population.rs:787-837 */
int pansim_group_run_generations_stats(pansim_group *g, uint32_t gen0, uint32_t n, const uint32_t *range1,
                                       const uint32_t *range2, size_t n_pairs, double *stats_out);
/* Exact all-pairs mode over the group (extension, BASELINE config 5): row blocks of about chunk_pairs
 * pairs; per block the partial core counts are reduce-scattered over the shards while the next block
 * is being computed. cb is called once per block, in (i, j) order; the vectors are valid during the
 * call; a non-zero return stops the walk and is returned. */
typedef int (*pansim_pairs_cb)(void *user, uint32_t row_begin, uint32_t row_end, size_t n_pairs,
                               const uint32_t *core_diff, const uint32_t *inter, const uint32_t *uni);
int pansim_group_all_pairs(pansim_group *g, size_t chunk_pairs, pansim_pairs_cb cb, void *user);
/* last walk: wall time (callbacks included), device time of shard 0 inside the reduce-scatters, pairs walked */
int pansim_group_all_pairs_timing(pansim_group *g, float *wall_ms, float *nccl_ms, uint64_t *pairs);
int pansim_group_gene_counts(pansim_group *g, uint32_t *counts);                          /* population.rs:840-856 */
/* whole-alignment diversity: the shard partials summed on the host (sfs [N+1] or NULL) */
int pansim_group_core_diversity(pansim_group *g, pansim_diversity *out, uint64_t *sfs);
int pansim_group_run_generations_diversity(pansim_group *g, uint32_t gen0, uint32_t n, const uint32_t *range1,
                                           const uint32_t *range2, size_t n_pairs, double *stats_out,
                                           pansim_diversity *div_out);
int pansim_group_download_acc(pansim_group *g, uint8_t *acc_out);
int pansim_group_download_core(pansim_group *g, uint8_t *core_onehot_out);               /* [N x core_size] */
int pansim_group_export_core_csv(pansim_group *g, uint32_t row_begin, uint32_t row_end, char *out);
/* the whole-alignment VCF of pansim_write_core_vcf: the header once, then every shard's lines in shard order */
int pansim_group_write_core_vcf(pansim_group *g, const char *path, uint64_t *bytes_out);
/* the whole-alignment FASTA of pansim_write_core_fasta, by row blocks: every shard's letters, the records written
 * on the host; columns and constant-site counts are the sums over the shards */
int pansim_group_write_core_fasta(pansim_group *g, const char *path, int snps_only, uint64_t *columns_out, uint64_t *const_counts, uint64_t *bytes_out);

/* pansim_core_ld over the whole alignment: every shard with the next one as its halo, summed on the host */
int pansim_group_core_ld(pansim_group *g, const pansim_ld_params *p, pansim_ld_bin *bins, uint64_t *sites_used);

/* pansim_gene_ld of the group: the accessory matrix is replicated in every shard, so shard 0 answers. Under a
 * communicator every rank computes the same whole result; nothing is exchanged. */
int pansim_group_gene_ld(pansim_group *g, const pansim_gene_ld_params *p, pansim_gene_ld_class classes[3],
                         uint64_t *hist, uint64_t genes_used[2]);

/* pansim_gene_accumulation and pansim_gene_spectrum of the group: the accessory matrix is replicated, so shard 0
 * answers. Under a communicator every rank computes the same whole result; nothing is exchanged. */
int pansim_group_gene_accumulation(pansim_group *g, uint64_t seed, uint32_t n_perms, uint32_t *orders, uint32_t *pan,
                                   uint32_t *core, uint32_t *new_genes, uint32_t *unique);
int pansim_group_gene_spectrum(pansim_group *g, uint64_t *spectrum);

/* the clonal genealogy of the group: every shard draws the same parents, so shard 0 records and answers. Under a
 * communicator (one process per GPU) every rank records its own identical copy; nothing is exchanged. */
int pansim_group_enable_genealogy(pansim_group *g, uint32_t capacity);
int pansim_group_genealogy(pansim_group *g, pansim_genealogy_node *nodes, pansim_genealogy_info *info);
int pansim_group_genealogy_tmrca(pansim_group *g, const uint32_t *r1, const uint32_t *r2, size_t n_pairs, uint32_t *tmrca);

/* parsimony of the group on a node table over its rows. Core: every shard answers for its columns; the summaries and
 * branch changes are summed and site_changes holds the shards' sites concatenated in shard (= site) order. Genes: the
 * accessory matrix is replicated, so shard 0 answers. Under a communicator a rank covers its own columns, as
 * pansim_core_ld does; nothing is exchanged. */
int pansim_group_core_parsimony(pansim_group *g, const uint32_t *parent, uint32_t n_nodes, pansim_parsimony *out,
                                uint32_t *site_changes, uint64_t *branch_changes);
int pansim_group_gene_parsimony(pansim_group *g, const uint32_t *parent, uint32_t n_nodes, pansim_parsimony *out,
                                uint32_t *gene_changes, uint64_t *gains, uint64_t *losses);
/* neighbour-joining tree of the group (pansim_nj_tree). Core: every shard counts its columns per row block, the counts
 * are summed over the shards (ncclAllReduce) and shard 0 builds the matrix and joins. Acc: the accessory matrix is
 * replicated, so shard 0 answers. Bit-identical to one context. */
int pansim_group_nj_tree(pansim_group *g, int metric, uint32_t *parent, double *length);

/* ---- introspection / instrumentation ----------------------------------- */
typedef struct {
    uint64_t core_row_stride_bytes;   /* packed row pitch on the device              */
    uint64_t acc_row_stride_bytes;
    uint64_t local_sites;             /* site_end - site_begin                       */
    uint64_t core_state_bytes;        /* one of the two packed core buffers          */
    uint64_t algorithmic_bytes_per_generation;  /* 2*N*ceil(Ll/4) + 2*N*ceil(G/8)   */
    uint64_t algorithmic_bytes_per_pair;        /* 2*ceil(Ll/4) + 2*ceil(G/8)       */
    uint32_t sm_count;
    uint32_t core_step_grid, core_step_block, core_step_smem;
} pansim_info;
int pansim_get_info(pansim_ctx *ctx, pansim_info *out);

/* Device time (ms, CUDA events on the context's stream) of the last
 * pansim_step / pansim_step_with_parents / pansim_run_generations /
 * pansim_pair_counts* call, split by kernel group. After pansim_core_diversity
 * total_ms is the reduction kernel alone (the diversity batches time like the
 * other batches). */
typedef struct {
    float total_ms;
    float core_step_ms;       /* core genome: gather+SNP kernel and the recombination pass (sum over generations) */
    float acc_step_ms;
    float select_ms;          /* competition + fitness + parent draw               */
    float pair_core_ms, pair_acc_ms;
    uint32_t launches;        /* kernels launched by that call                     */
    float core_hr_ms;         /* the recombination pass alone (part of core_step_ms) */
} pansim_timing;
int pansim_get_timing(pansim_ctx *ctx, pansim_timing *out);
/* enable/disable per-kernel event timing (off = no extra events; default on) */
int pansim_set_timing(pansim_ctx *ctx, int enabled);

/* Generate-mode event dump for parity tests: when enabled, the next
 * pansim_step* call also records every event it draws, so the oracle can
 * replay them with the reference's semantics. seq = order among events of one
 * (row, site block); the per-cell winner is the highest seq. */
typedef struct {
    size_t n_core_mut;  uint32_t *core_mut_row, *core_mut_site, *core_mut_seq; uint8_t *core_mut_allele;
    size_t n_hr;        uint32_t *hr_recipient, *hr_locus, *hr_donor, *hr_seq;  uint8_t *hr_value;
    uint8_t *acc_flip_mask;   /* [N x G] 1 = flipped (population.rs:504-508 parity) */
    uint8_t *acc_gain_mask;   /* [N x G] 1 = received by HGT                        */
} pansim_event_dump;
int  pansim_enable_event_dump(pansim_ctx *ctx, size_t max_core_events);
/* arrays are malloc'd by the library; release with pansim_free_event_dump */
int  pansim_fetch_event_dump(pansim_ctx *ctx, pansim_event_dump *out);
void pansim_free_event_dump(pansim_event_dump *d);

/* per-cell probabilities the generate-mode kernels use (documentation of the
 * thinning, SURVEY.md 8a rows M and R); out has 4 doubles:
 * [0] core site overwritten by U{C,G,T} per generation, [1] core cell
 * overwritten by a donor allele, [2],[3] accessory flip prob. compartment 0,1 */
int pansim_get_rates(pansim_ctx *ctx, double *out);

#ifdef __cplusplus
}
#endif
#endif /* PANSIM_B200_H */
