"""ctypes binding of libpansim_b200.so (include/pansim_b200.h).

Plumbing only: loads the in-tree shared library built by pansim_b200/csrc/Makefile
and declares the C signatures. There is no fallback: if the library is missing
or no B200 is present the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PANSIM_B200_LIB") or os.path.join(_HERE, "libpansim_b200.so")   # override: kernel-variant experiments

EXPORTED = [
    "pansim_config_init", "pansim_create", "pansim_destroy", "pansim_last_error", "pansim_version",
    "pansim_set_initial", "pansim_upload_core", "pansim_upload_acc", "pansim_download_core",
    "pansim_download_acc", "pansim_export_core_csv", "pansim_set_selection",
    "pansim_average_distance", "pansim_sample_indices", "pansim_get_weights",
    "pansim_step_with_parents", "pansim_step", "pansim_run_generations", "pansim_next_generation",
    "pansim_get_parents", "pansim_step_replay", "pansim_pair_counts", "pansim_pair_counts_device",
    "pansim_pair_counts_rows", "pansim_pair_counts_rows_device",
    "pansim_core_distance", "pansim_acc_distance", "pansim_gene_counts", "pansim_get_info",
    "pansim_get_timing", "pansim_set_timing", "pansim_enable_event_dump",
    "pansim_fetch_event_dump", "pansim_free_event_dump", "pansim_get_rates",
    "pansim_select_parents", "pansim_pair_stats", "pansim_run_generations_stats", "pansim_write_core_csv",
    "pansim_comm_unique_id", "pansim_comm_init_rank", "pansim_comm_info",
    "pansim_shard_bounds", "pansim_group_create", "pansim_group_destroy", "pansim_group_last_error", "pansim_group_size", "pansim_group_ctx",
    "pansim_group_set_initial", "pansim_group_set_selection", "pansim_group_run_generations", "pansim_group_pair_counts",
    "pansim_group_run_generations_stats", "pansim_group_all_pairs", "pansim_group_all_pairs_timing", "pansim_group_gene_counts",
    "pansim_group_download_acc", "pansim_group_download_core", "pansim_group_export_core_csv",
    "pansim_core_allele_counts", "pansim_core_diversity", "pansim_run_generations_diversity", "pansim_diversity_stats",
    "pansim_group_core_diversity", "pansim_group_run_generations_diversity",
    "pansim_write_core_vcf", "pansim_group_write_core_vcf", "pansim_core_vcf_kernel_ms",
    "pansim_write_core_fasta", "pansim_export_core_fasta_rows", "pansim_group_write_core_fasta", "pansim_core_fasta_kernel_ms",
    "pansim_core_ld", "pansim_group_core_ld", "pansim_core_ld_kernel_ms", "pansim_ld_mean_r2",
    "pansim_gene_ld", "pansim_group_gene_ld", "pansim_gene_ld_kernel_ms",
    "pansim_gene_accumulation", "pansim_group_gene_accumulation", "pansim_gene_accumulation_kernel_ms",
    "pansim_gene_spectrum", "pansim_group_gene_spectrum", "pansim_pangenome_classes",
    "pansim_core_parsimony", "pansim_gene_parsimony", "pansim_parsimony_kernel_ms", "pansim_parsimony_indices",
    "pansim_group_core_parsimony", "pansim_group_gene_parsimony",
    "pansim_nj_tree", "pansim_nj_tree_matrix", "pansim_nj_kernel_ms", "pansim_tree_newick", "pansim_tree_compare_splits",
    "pansim_group_nj_tree",
    "pansim_enable_genealogy", "pansim_genealogy", "pansim_genealogy_history", "pansim_genealogy_tmrca",
    "pansim_genealogy_newick", "pansim_group_enable_genealogy", "pansim_group_genealogy", "pansim_group_genealogy_tmrca",
]
COMM_ID_BYTES = 128


class Config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("device", C.c_int32), ("pop_size", C.c_uint32),
        ("pan_size", C.c_uint32), ("core_size", C.c_uint64), ("site_begin", C.c_uint64),
        ("site_end", C.c_uint64), ("core_genes", C.c_uint32), ("n_compartments", C.c_uint32),
        ("comp_lo", C.c_uint32 * 2), ("comp_hi", C.c_uint32 * 2), ("core_mut_mean", C.c_double),
        ("hr_mean", C.c_double), ("acc_mut_mean", C.c_double * 2), ("hgt_mean", C.c_double * 2),
        ("avg_gene_num", C.c_int32), ("no_control_genome_size", C.c_int32),
        ("genome_size_penalty", C.c_double), ("competition_strength", C.c_double),
        ("seed", C.c_uint64),
    ]


class Events(C.Structure):
    _fields_ = [
        ("parents", C.c_void_p),
        ("n_core_mut", C.c_size_t), ("core_mut_row", C.c_void_p), ("core_mut_site", C.c_void_p),
        ("core_mut_allele", C.c_void_p),
        ("n_acc_flip", C.c_size_t), ("acc_flip_row", C.c_void_p), ("acc_flip_gene", C.c_void_p),
        ("n_hr", C.c_size_t), ("hr_recipient", C.c_void_p), ("hr_locus", C.c_void_p),
        ("hr_value", C.c_void_p),
        ("n_hgt", C.c_size_t), ("hgt_recipient", C.c_void_p), ("hgt_gene", C.c_void_p),
    ]


class Info(C.Structure):
    _fields_ = [
        ("core_row_stride_bytes", C.c_uint64), ("acc_row_stride_bytes", C.c_uint64),
        ("local_sites", C.c_uint64), ("core_state_bytes", C.c_uint64),
        ("algorithmic_bytes_per_generation", C.c_uint64), ("algorithmic_bytes_per_pair", C.c_uint64),
        ("sm_count", C.c_uint32), ("core_step_grid", C.c_uint32), ("core_step_block", C.c_uint32),
        ("core_step_smem", C.c_uint32),
    ]


class Timing(C.Structure):
    _fields_ = [
        ("total_ms", C.c_float), ("core_step_ms", C.c_float), ("acc_step_ms", C.c_float),
        ("select_ms", C.c_float), ("pair_core_ms", C.c_float), ("pair_acc_ms", C.c_float),
        ("launches", C.c_uint32), ("core_hr_ms", C.c_float),
    ]


class EventDump(C.Structure):
    _fields_ = [
        ("n_core_mut", C.c_size_t), ("core_mut_row", C.POINTER(C.c_uint32)),
        ("core_mut_site", C.POINTER(C.c_uint32)), ("core_mut_seq", C.POINTER(C.c_uint32)),
        ("core_mut_allele", C.POINTER(C.c_uint8)),
        ("n_hr", C.c_size_t), ("hr_recipient", C.POINTER(C.c_uint32)),
        ("hr_locus", C.POINTER(C.c_uint32)), ("hr_donor", C.POINTER(C.c_uint32)),
        ("hr_seq", C.POINTER(C.c_uint32)), ("hr_value", C.POINTER(C.c_uint8)),
        ("acc_flip_mask", C.POINTER(C.c_uint8)), ("acc_gain_mask", C.POINTER(C.c_uint8)),
    ]


class Diversity(C.Structure):
    _fields_ = [("sites", C.c_uint64), ("segregating", C.c_uint64), ("multiallelic", C.c_uint64),
                ("pair_diff_sum", C.c_uint64)]


class LdParams(C.Structure):
    _fields_ = [("max_dist", C.c_uint32), ("bin_width", C.c_uint32), ("min_minor", C.c_uint32)]


class LdBin(C.Structure):
    _fields_ = [("pairs", C.c_uint64), ("four_gamete", C.c_uint64), ("r2_hi", C.c_uint64), ("r2_lo", C.c_uint64)]


class GeneLdParams(C.Structure):
    _fields_ = [("r2_bins", C.c_uint32), ("min_minor", C.c_uint32)]


class GeneLdClass(C.Structure):
    _fields_ = [("ld", LdBin), ("associated", C.c_uint64), ("dissociated", C.c_uint64)]


class Parsimony(C.Structure):
    _fields_ = [("characters", C.c_uint64), ("variable", C.c_uint64), ("tree_length", C.c_uint64),
                ("min_changes", C.c_uint64), ("max_changes", C.c_uint64), ("homoplastic", C.c_uint64)]


class GenealogyNode(C.Structure):
    _fields_ = [("parent", C.c_uint32), ("individual", C.c_uint32), ("time", C.c_uint32)]


class GenealogyInfo(C.Structure):
    _fields_ = [("generations_total", C.c_uint64), ("generations_kept", C.c_uint32), ("n_nodes", C.c_uint32),
                ("lineages_at_start", C.c_uint32)]


PAIRS_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t, C.POINTER(C.c_uint32),
                       C.POINTER(C.c_uint32), C.POINTER(C.c_uint32))


def build(force: bool = False) -> str:
    """Compile libpansim_b200.so for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    src_dir = os.path.join(_HERE, "csrc")
    srcs = [os.path.join(src_dir, f) for f in os.listdir(src_dir) if f.endswith((".cu", ".cuh", ".hpp", ".inl"))]
    srcs.append(os.path.join(_HERE, "..", "include", "pansim_b200.h"))
    stale = (not os.path.exists(LIB_PATH)) or any(
        os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs if os.path.exists(s))
    if force or stale:
        subprocess.run(["make", "-C", src_dir] + (["-B"] if force else []), check=True,
                       stdout=subprocess.DEVNULL)
    return LIB_PATH


_lib = None


def lib():
    """Load the shared library (building it if the sources are newer)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        try:
            build()
        except Exception as e:  # no nvcc on this box: fail loudly, never fall back
            raise RuntimeError(
                f"{LIB_PATH} is missing and could not be built ({e}); "
                "pansim_b200 has no CPU fallback") from e
    L = C.CDLL(LIB_PATH)
    vp, sz, u32, dbl, cint = C.c_void_p, C.c_size_t, C.c_uint32, C.c_double, C.c_int

    def sig(name, res, *args):
        f = getattr(L, name)
        f.restype = res
        f.argtypes = list(args)

    sig("pansim_config_init", None, C.POINTER(Config))
    sig("pansim_create", cint, C.POINTER(Config), C.POINTER(vp))
    sig("pansim_destroy", None, vp)
    sig("pansim_last_error", C.c_char_p, vp)
    sig("pansim_version", C.c_char_p)
    sig("pansim_set_initial", cint, vp, vp, vp)
    sig("pansim_upload_core", cint, vp, vp)
    sig("pansim_upload_acc", cint, vp, vp)
    sig("pansim_download_core", cint, vp, vp)
    sig("pansim_download_acc", cint, vp, vp)
    sig("pansim_export_core_csv", cint, vp, u32, u32, vp)
    sig("pansim_set_selection", cint, vp, vp)
    sig("pansim_average_distance", cint, vp, vp)
    sig("pansim_sample_indices", cint, vp, u32, vp, vp)
    sig("pansim_get_weights", cint, vp, vp, vp, vp)
    sig("pansim_step_with_parents", cint, vp, u32, vp)
    sig("pansim_step", cint, vp, u32)
    sig("pansim_run_generations", cint, vp, u32, u32)
    sig("pansim_next_generation", cint, vp, vp)
    sig("pansim_get_parents", cint, vp, vp)
    sig("pansim_step_replay", cint, vp, C.POINTER(Events))
    sig("pansim_pair_counts", cint, vp, vp, vp, sz, vp, vp, vp)
    sig("pansim_pair_counts_device", cint, vp, vp, vp, sz, vp, vp, vp)
    sig("pansim_pair_counts_rows", cint, vp, u32, u32, vp, vp, vp, vp)
    sig("pansim_pair_counts_rows_device", cint, vp, u32, u32, vp, vp, vp, vp)
    sig("pansim_core_distance", dbl, u32, C.c_uint64)
    sig("pansim_acc_distance", dbl, u32, u32, u32)
    sig("pansim_gene_counts", cint, vp, vp)
    sig("pansim_get_info", cint, vp, C.POINTER(Info))
    sig("pansim_get_timing", cint, vp, C.POINTER(Timing))
    sig("pansim_set_timing", cint, vp, cint)
    sig("pansim_enable_event_dump", cint, vp, sz)
    sig("pansim_fetch_event_dump", cint, vp, C.POINTER(EventDump))
    sig("pansim_free_event_dump", None, C.POINTER(EventDump))
    sig("pansim_get_rates", cint, vp, vp)
    sig("pansim_select_parents", cint, vp, u32, vp, vp)
    sig("pansim_write_core_csv", cint, vp, C.c_char_p, C.POINTER(C.c_uint64))
    sig("pansim_pair_stats", cint, vp, vp, vp, sz, vp)
    sig("pansim_run_generations_stats", cint, vp, u32, u32, vp, vp, sz, vp)
    sig("pansim_comm_unique_id", cint, vp)
    sig("pansim_comm_init_rank", cint, vp, cint, cint, vp)
    sig("pansim_comm_info", cint, vp, C.POINTER(cint), C.POINTER(cint))
    sig("pansim_shard_bounds", cint, C.c_uint64, cint, cint, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64))
    sig("pansim_group_create", cint, C.POINTER(Config), cint, vp, C.POINTER(vp))
    sig("pansim_group_destroy", None, vp)
    sig("pansim_group_last_error", C.c_char_p, vp)
    sig("pansim_group_size", cint, vp)
    sig("pansim_group_ctx", vp, vp, cint)
    sig("pansim_group_set_initial", cint, vp, vp, vp)
    sig("pansim_group_set_selection", cint, vp, vp)
    sig("pansim_group_run_generations", cint, vp, u32, u32)
    sig("pansim_group_pair_counts", cint, vp, vp, vp, sz, vp, vp, vp)
    sig("pansim_group_run_generations_stats", cint, vp, u32, u32, vp, vp, sz, vp)
    sig("pansim_group_all_pairs", cint, vp, sz, PAIRS_CB, vp)
    sig("pansim_group_all_pairs_timing", cint, vp, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_uint64))
    sig("pansim_group_gene_counts", cint, vp, vp)
    sig("pansim_group_download_acc", cint, vp, vp)
    sig("pansim_group_download_core", cint, vp, vp)
    sig("pansim_group_export_core_csv", cint, vp, u32, u32, vp)
    sig("pansim_core_allele_counts", cint, vp, vp)
    sig("pansim_core_diversity", cint, vp, C.POINTER(Diversity), vp)
    sig("pansim_run_generations_diversity", cint, vp, u32, u32, vp, vp, sz, vp, vp)
    sig("pansim_diversity_stats", None, C.POINTER(Diversity), u32, vp)
    sig("pansim_group_core_diversity", cint, vp, C.POINTER(Diversity), vp)
    sig("pansim_group_run_generations_diversity", cint, vp, u32, u32, vp, vp, sz, vp, vp)
    sig("pansim_write_core_vcf", cint, vp, C.c_char_p, cint, C.POINTER(C.c_uint64))
    sig("pansim_group_write_core_vcf", cint, vp, C.c_char_p, C.POINTER(C.c_uint64))
    sig("pansim_core_vcf_kernel_ms", cint, vp, u32, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_uint64))
    sig("pansim_write_core_fasta", cint, vp, C.c_char_p, cint, C.POINTER(C.c_uint64), vp, C.POINTER(C.c_uint64))
    sig("pansim_export_core_fasta_rows", cint, vp, cint, u32, u32, vp, C.POINTER(C.c_uint64))
    sig("pansim_group_write_core_fasta", cint, vp, C.c_char_p, cint, C.POINTER(C.c_uint64), vp, C.POINTER(C.c_uint64))
    sig("pansim_core_fasta_kernel_ms", cint, vp, cint, u32, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_uint64))
    sig("pansim_core_ld", cint, vp, vp, C.POINTER(LdParams), C.POINTER(LdBin), C.POINTER(C.c_uint64))
    sig("pansim_group_core_ld", cint, vp, C.POINTER(LdParams), C.POINTER(LdBin), C.POINTER(C.c_uint64))
    sig("pansim_core_ld_kernel_ms", cint, vp, C.POINTER(LdParams), u32, C.POINTER(C.c_float), C.POINTER(C.c_float),
        C.POINTER(C.c_float), C.POINTER(C.c_uint64))
    sig("pansim_ld_mean_r2", dbl, C.POINTER(LdBin))
    sig("pansim_gene_ld", cint, vp, C.POINTER(GeneLdParams), C.POINTER(GeneLdClass), vp, vp)
    sig("pansim_group_gene_ld", cint, vp, C.POINTER(GeneLdParams), C.POINTER(GeneLdClass), vp, vp)
    sig("pansim_gene_ld_kernel_ms", cint, vp, C.POINTER(GeneLdParams), u32, C.POINTER(C.c_float), C.POINTER(C.c_float),
        C.POINTER(C.c_float), C.POINTER(C.c_uint64))
    sig("pansim_gene_accumulation", cint, vp, C.c_uint64, u32, vp, vp, vp, vp, vp)
    sig("pansim_group_gene_accumulation", cint, vp, C.c_uint64, u32, vp, vp, vp, vp, vp)
    sig("pansim_gene_accumulation_kernel_ms", cint, vp, C.c_uint64, u32, u32, C.POINTER(C.c_float), C.POINTER(C.c_float),
        C.POINTER(C.c_uint64))
    sig("pansim_gene_spectrum", cint, vp, vp)
    sig("pansim_group_gene_spectrum", cint, vp, vp)
    sig("pansim_pangenome_classes", None, vp, u32, vp)
    sig("pansim_core_parsimony", cint, vp, vp, u32, C.POINTER(Parsimony), vp, vp)
    sig("pansim_gene_parsimony", cint, vp, vp, u32, C.POINTER(Parsimony), vp, vp, vp)
    sig("pansim_group_core_parsimony", cint, vp, vp, u32, C.POINTER(Parsimony), vp, vp)
    sig("pansim_group_gene_parsimony", cint, vp, vp, u32, C.POINTER(Parsimony), vp, vp, vp)
    sig("pansim_parsimony_kernel_ms", cint, vp, vp, u32, cint, u32, C.POINTER(C.c_float), C.POINTER(C.c_uint64),
        C.POINTER(C.c_uint32))
    sig("pansim_parsimony_indices", None, C.POINTER(Parsimony), C.POINTER(C.c_double), C.POINTER(C.c_double))
    sig("pansim_nj_tree", cint, vp, cint, vp, vp)
    sig("pansim_group_nj_tree", cint, vp, cint, vp, vp)
    sig("pansim_nj_tree_matrix", cint, vp, vp, u32, vp, vp)
    sig("pansim_nj_kernel_ms", cint, vp, cint, u32, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_uint64),
        C.POINTER(C.c_uint32))
    sig("pansim_tree_newick", cint, vp, vp, u32, u32, vp, sz, C.POINTER(sz))
    sig("pansim_tree_compare_splits", cint, vp, u32, vp, u32, u32, vp)
    sig("pansim_enable_genealogy", cint, vp, u32)
    sig("pansim_genealogy", cint, vp, vp, C.POINTER(GenealogyInfo))
    sig("pansim_genealogy_history", cint, vp, vp)
    sig("pansim_genealogy_tmrca", cint, vp, vp, vp, sz, vp)
    sig("pansim_genealogy_newick", cint, vp, u32, u32, vp, sz, C.POINTER(sz))
    sig("pansim_group_enable_genealogy", cint, vp, u32)
    sig("pansim_group_genealogy", cint, vp, vp, C.POINTER(GenealogyInfo))
    sig("pansim_group_genealogy_tmrca", cint, vp, vp, vp, sz, vp)
    _lib = L
    return L
