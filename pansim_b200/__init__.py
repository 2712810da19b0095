"""pansim_b200: B200 (sm_100a) implementation of Pansim's per-generation
Wright-Fisher step and pairwise distance pass, behind a C ABI
(include/pansim_b200.h, libpansim_b200.so) with a thin ctypes host mirror of the
reference's `Population` API. No CPU fallback."""
from .params import Derived, Params, derive, fmt_f64, validate  # noqa: F401
from .population import (CoreFasta, CoreLD, CoreParsimony, Diversity, GeneAccumulation, GeneLD, GeneParsimony,  # noqa: F401
                         Genealogy, NJTree, Pansim, PansimError, SplitComparison, compare_splits, diversity_stats,
                         genealogy_newick, make_config, pangenome_classes, parsimony_indices, standard_deviation,
                         tree_newick)
from .group import PansimGroup  # noqa: F401

__version__ = "0.1.0"
