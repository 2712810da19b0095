"""Host-side mirror of the reference's `Population` API over the C ABI.

`Pansim` owns one `pansim_ctx` = the reference's `core_genome` + `pan_genome`
pair (main.rs:372-391), because the reference always moves them together with
the same parent vector (main.rs:442-464). Method names follow
pansim/src/population.rs; argument meaning and error behaviour are documented
per method. numpy arrays are host buffers; nothing here computes on the CPU
except the f64 divisions the reference also does on the host side of the
boundary (population.rs:822, 828-830, 852).
"""
from __future__ import annotations

import ctypes as C
from typing import NamedTuple

import numpy as np

from . import _ffi
from .params import Derived, Params, derive, fmt_f64

OK = 0


class PansimError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"[{code}] {msg}")
        self.code = code


def _ptr(a: np.ndarray | None):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def make_config(p: Params, d: Derived | None = None, device: int = 0, site_begin: int = 0,
                site_end: int = 0) -> _ffi.Config:
    """pansim_config from the command-line parameters (main.rs:259-287, 333-367)."""
    d = d or derive(p)
    cfg = _ffi.Config()
    _ffi.lib().pansim_config_init(C.byref(cfg))
    cfg.device = device
    cfg.pop_size = p.pop_size
    cfg.pan_size = d.pan_size
    cfg.core_size = p.core_size
    cfg.site_begin, cfg.site_end = site_begin, site_end
    cfg.core_genes = p.core_genes
    cfg.n_compartments = len(d.comp)
    for k, (lo, hi) in enumerate(d.comp):
        cfg.comp_lo[k], cfg.comp_hi[k] = lo, hi
        cfg.acc_mut_mean[k] = d.n_pan_mutations[k]
        cfg.hgt_mean[k] = d.n_recombinations_pan[k] if p.HGT_rate > 0.0 else 0.0   # main.rs:462
    cfg.core_mut_mean = d.n_core_mutations
    cfg.hr_mean = d.n_recombinations_core if p.HR_rate > 0.0 else 0.0              # main.rs:459
    cfg.avg_gene_num = d.avg_gene_num
    cfg.no_control_genome_size = int(p.no_control_genome_size)
    cfg.genome_size_penalty = p.genome_size_penalty
    cfg.competition_strength = p.competition_strength
    cfg.seed = p.seed
    return cfg


def standard_deviation(values) -> tuple[float, float]:
    """population.rs:87-94: (std, mean) with sequential f64 sums (np.cumsum is a
    sequential scan, unlike np.sum's pairwise reduction)."""
    v = np.ascontiguousarray(values, np.float64)
    n = len(v)
    mean = float(np.cumsum(v)[-1]) / n
    d = v - mean
    ss = float(np.cumsum(d * d)[-1])
    return float(np.sqrt(ss / n)), mean


class Diversity(NamedTuple):
    """pansim_diversity: integer summaries of the core alignment (partials over the sites of a column shard)."""
    sites: int
    segregating: int
    multiallelic: int
    pair_diff_sum: int


def _diversity(d: _ffi.Diversity) -> Diversity:
    return Diversity(d.sites, d.segregating, d.multiallelic, d.pair_diff_sum)


def diversity_stats(d: Diversity, pop_size: int) -> tuple[float, float, float]:
    """(pi, theta_W, Tajima's D) of whole-alignment summaries, evaluated by the library (pansim_diversity_stats)
    so every host forms the same bits. D is NaN when no site segregates; all three are NaN when pop_size < 2."""
    out = np.empty(3, np.float64)
    _ffi.lib().pansim_diversity_stats(C.byref(_ffi.Diversity(*d)), pop_size, _ptr(out))
    return float(out[0]), float(out[1]), float(out[2])


class CoreFasta(NamedTuple):
    """What a FASTA writer wrote (include/pansim_b200.h): bytes of the file, columns per record and, for the sites
    that are not columns, how many carry A, C, G and T (all 0 in whole mode; IQ-TREE's -fconst in SNP mode)."""
    bytes: int
    columns: int
    const_counts: np.ndarray


def _write_fasta(call, check, path: str, snps_only: bool) -> CoreFasta:
    cols, n = C.c_uint64(0), C.c_uint64(0)
    consts = np.zeros(4, np.uint64)
    check(call(path.encode(), int(snps_only), C.byref(cols), _ptr(consts), C.byref(n)))
    return CoreFasta(n.value, cols.value, consts)


class CoreLD(NamedTuple):
    """LD bins of pansim_core_ld (include/pansim_b200.h): per bin its distances dist_lo..dist_hi, the site pairs, the
    pairs showing four gametes, the exact sum of r^2 in units of 2^-32 and the mean r^2 (NaN for an empty bin); and
    the used sites counted."""
    dist_lo: np.ndarray
    dist_hi: np.ndarray
    pairs: np.ndarray
    four_gamete: np.ndarray
    r2_sum: list
    mean_r2: np.ndarray
    sites_used: int


def _ld_params(max_dist: int, bin_width: int, min_minor: int) -> _ffi.LdParams:
    return _ffi.LdParams(max_dist, bin_width, min_minor)


def _ld_bins(max_dist: int, bin_width: int):
    n = -(-max_dist // bin_width) if max_dist > 0 and bin_width > 0 else 1
    return (_ffi.LdBin * max(n, 1))(), n


def _core_ld(bins, n: int, max_dist: int, bin_width: int, used: int) -> CoreLD:
    lib = _ffi.lib()
    lo = np.arange(n, dtype=np.int64) * bin_width + 1
    hi = np.minimum(lo + bin_width - 1, max_dist)
    return CoreLD(lo, hi, np.array([b.pairs for b in bins[:n]], np.uint64),
                  np.array([b.four_gamete for b in bins[:n]], np.uint64),
                  [(b.r2_hi << 64) | b.r2_lo for b in bins[:n]],
                  np.array([lib.pansim_ld_mean_r2(C.byref(b)) for b in bins[:n]], np.float64), used)


def ld_mean_r2(pairs: int, r2_sum: int) -> float:
    """Mean r^2 of a bin from its pair count and exact r^2 sum (units of 2^-32), formed by the library."""
    return _ffi.lib().pansim_ld_mean_r2(C.byref(_ffi.LdBin(pairs, 0, r2_sum >> 64, r2_sum & (2 ** 64 - 1))))


GENE_LD_CLASSES = ("0-0", "0-1", "1-1")


class GeneLD(NamedTuple):
    """Accessory-gene linkage of pansim_gene_ld (include/pansim_b200.h), one entry per class of gene pair in the order
    of `classes` (the groups of the two genes: 0-0, 0-1, 1-1): the gene pairs, those showing four gametes, the
    associated (D > 0) and dissociated (D < 0) ones, the exact sum of r^2 in units of 2^-32 and the mean r^2 (NaN for
    an empty class); hist [3, r2_bins] the pairs per r^2 bin, and genes_used [2] the used genes of each group."""
    classes: tuple
    pairs: np.ndarray
    four_gamete: np.ndarray
    associated: np.ndarray
    dissociated: np.ndarray
    r2_sum: list
    mean_r2: np.ndarray
    hist: np.ndarray
    genes_used: np.ndarray


def _gene_ld(call, check, r2_bins: int, min_minor: int) -> GeneLD:
    """call(params, classes, hist, genes_used) -> status; the histogram is only allocated for a valid r2_bins (the
    library refuses the others before writing)."""
    cls = (_ffi.GeneLdClass * 3)()
    hist = np.zeros((3, r2_bins if 1 <= r2_bins <= 1024 else 0), np.uint64)
    used = np.zeros(2, np.uint64)
    check(call(C.byref(_ffi.GeneLdParams(r2_bins, min_minor)), cls, _ptr(hist) if hist.size else None, _ptr(used)))
    lib = _ffi.lib()
    return GeneLD(GENE_LD_CLASSES, np.array([c.ld.pairs for c in cls], np.uint64),
                  np.array([c.ld.four_gamete for c in cls], np.uint64), np.array([c.associated for c in cls], np.uint64),
                  np.array([c.dissociated for c in cls], np.uint64), [(c.ld.r2_hi << 64) | c.ld.r2_lo for c in cls],
                  np.array([lib.pansim_ld_mean_r2(C.byref(c.ld)) for c in cls], np.float64), hist, used)


GENE_ACC_MAX_PERMS = 10000      # PANSIM_GENE_ACC_MAX_PERMS


class GeneAccumulation(NamedTuple):
    """Pangenome accumulation curves of pansim_gene_accumulation (include/pansim_b200.h), each uint32 [P, N]: the
    random orders of the rows, and per order and number of genomes k = 1..N the pan genes, the core (conserved)
    genes, the new genes and the unique genes (Roary's four .Rtab curves). The core_genes count in pan and core at
    every k, and in new and unique at k = 1."""
    orders: np.ndarray
    pan: np.ndarray
    core: np.ndarray
    new: np.ndarray
    unique: np.ndarray


def _gene_accumulation(call, check, N: int, n_perms: int, seed: int) -> GeneAccumulation:
    """call(seed, n_perms, orders, pan, core, new, unique) -> status; the arrays are only sized for a valid n_perms
    (the library refuses the others before writing)."""
    P = n_perms if 1 <= n_perms <= GENE_ACC_MAX_PERMS else 0
    out = [np.empty((P, N), np.uint32) for _ in range(5)]
    check(call(seed, n_perms, *[_ptr(a) for a in out]))
    return GeneAccumulation(*out)


def _gene_spectrum(call, check, N: int) -> np.ndarray:
    out = np.empty(N + 1, np.uint64)
    check(call(_ptr(out)))
    return out


PANGENOME_CLASSES = ("core", "soft_core", "shell", "cloud", "total")


def pangenome_classes(spectrum, pop_size: int) -> tuple[int, int, int, int, int]:
    """(core, soft core, shell, cloud, total) genes of a gene frequency spectrum [pop_size + 1] by Roary's
    thresholds as integer tests, evaluated by the library (pansim_pangenome_classes) so every host prints the same."""
    spec = np.ascontiguousarray(spectrum, np.uint64)
    if spec.shape != (pop_size + 1,):
        raise ValueError(f"spectrum must have pop_size + 1 = {pop_size + 1} bins, not {spec.shape}")
    out = np.zeros(5, np.uint64)
    _ffi.lib().pansim_pangenome_classes(_ptr(spec), pop_size, _ptr(out))
    return tuple(int(x) for x in out)


PARSIMONY_FIELDS = ("characters", "variable", "tree_length", "min_changes", "max_changes", "homoplastic")


class CoreParsimony(NamedTuple):
    """Parsimony of the core sites on a node table (pansim_core_parsimony, include/pansim_b200.h): the summary, the
    consistency and retention indices (NaN for a zero denominator), the score of every local site (uint32, position
    order) and the changes on the branch above every node (uint64 [n_nodes], 0 at the root)."""
    characters: int
    variable: int
    tree_length: int
    min_changes: int
    max_changes: int
    homoplastic: int
    ci: float
    ri: float
    site_changes: np.ndarray
    branch_changes: np.ndarray


class GeneParsimony(NamedTuple):
    """Parsimony of the accessory genes on a node table (pansim_gene_parsimony): the summary, CI and RI, the score of
    every matrix gene (uint32, _pangenome.csv column order) and the gains and losses on the branch above every node
    (uint64 [n_nodes], 0 at the root)."""
    characters: int
    variable: int
    tree_length: int
    min_changes: int
    max_changes: int
    homoplastic: int
    ci: float
    ri: float
    gene_changes: np.ndarray
    gains: np.ndarray
    losses: np.ndarray


def parsimony_indices(summary) -> tuple[float, float]:
    """(CI, RI) = (M / S, (G - S) / (G - M)) of a parsimony summary (anything with the six summary fields), NaN for a
    zero denominator, evaluated by the library (pansim_parsimony_indices) so every host prints the same."""
    p = _ffi.Parsimony(*(int(getattr(summary, f)) for f in PARSIMONY_FIELDS))
    ci, ri = C.c_double(), C.c_double()
    _ffi.lib().pansim_parsimony_indices(C.byref(p), C.byref(ci), C.byref(ri))
    return ci.value, ri.value


def _parent_table(genealogy) -> np.ndarray:
    """The parent column of a Genealogy, or a parent array itself, as contiguous uint32."""
    parent = genealogy.parent if hasattr(genealogy, "parent") else genealogy
    return np.ascontiguousarray(parent, np.uint32)


def _parsimony(call, check, parent: np.ndarray, n_chars: int, genes: bool):
    """call(parent, n_nodes, &summary, chars, branch arrays...) -> status."""
    n = len(parent)
    s = _ffi.Parsimony()
    chars = np.zeros(n_chars, np.uint32)
    branches = [np.zeros(n, np.uint64) for _ in range(2 if genes else 1)]
    check(call(_ptr(parent), n, C.byref(s), _ptr(chars), *[_ptr(b) for b in branches]))
    head = tuple(int(getattr(s, f)) for f in PARSIMONY_FIELDS)
    ci, ri = parsimony_indices(s)
    return (GeneParsimony if genes else CoreParsimony)(*head, ci, ri, chars, *branches)


class Genealogy(NamedTuple):
    """The clonal genealogy of the present population (pansim_genealogy, include/pansim_b200.h): per node its parent
    (0xFFFFFFFF at the root), the individual it stands for (0xFFFFFFFF at a virtual root) and its time in generations
    before the present; leaves are nodes 0 .. n_leaves-1. generations_total vectors were recorded since the last
    reset, generations_kept of them are traced; lineages_at_start = 1 means the MRCA was found."""
    parent: np.ndarray
    individual: np.ndarray
    time: np.ndarray
    generations_total: int
    generations_kept: int
    n_nodes: int
    lineages_at_start: int
    n_leaves: int

    def newick(self) -> str:
        """The canonical Newick text (leaves `ind_<i>`, integer branch lengths), formatted by the library."""
        return genealogy_newick(self.parent, self.individual, self.time, self.n_leaves)


def genealogy_newick(parent, individual, time, n_leaves: int) -> str:
    """pansim_genealogy_newick of a node table given as three arrays (no device)."""
    lib = _ffi.lib()
    table = np.ascontiguousarray(np.stack([np.asarray(parent), np.asarray(individual), np.asarray(time)], axis=1), np.uint32)
    n = C.c_size_t(0)
    rc = lib.pansim_genealogy_newick(_ptr(table), len(table), n_leaves, None, 0, C.byref(n))
    if rc != OK:
        raise PansimError(rc, "pansim_genealogy_newick: not a tree of that shape")
    buf = C.create_string_buffer(n.value + 1)
    rc = lib.pansim_genealogy_newick(_ptr(table), len(table), n_leaves, buf, n.value + 1, C.byref(n))
    if rc != OK:
        raise PansimError(rc, "pansim_genealogy_newick failed")
    return buf.raw[:n.value].decode()


NJ_METRICS = {"core": 0, "acc": 1}


def nj_nodes(n_leaves: int) -> int:
    """Nodes of a neighbour-joining table over n_leaves leaves: 2N - 2 for N >= 3, 3 for N = 2, 1 for N = 1."""
    return 2 * n_leaves - 2 if n_leaves >= 3 else 3 if n_leaves == 2 else 1


def tree_newick(parent, length, n_leaves: int) -> str:
    """pansim_tree_newick of a node table with branch lengths (no device): leaves ind_<i>, children ordered by their
    smallest leaf, lengths %.17g."""
    lib = _ffi.lib()
    parent = np.ascontiguousarray(parent, np.uint32)
    length = np.ascontiguousarray(length, np.float64)
    if len(length) != len(parent):
        raise ValueError("parent and length differ in length")
    n = C.c_size_t(0)
    rc = lib.pansim_tree_newick(_ptr(parent), _ptr(length), len(parent), n_leaves, None, 0, C.byref(n))
    if rc != OK:
        raise PansimError(rc, "pansim_tree_newick: not a node table over that many leaves")
    buf = C.create_string_buffer(n.value + 1)
    rc = lib.pansim_tree_newick(_ptr(parent), _ptr(length), len(parent), n_leaves, buf, n.value + 1, C.byref(n))
    if rc != OK:
        raise PansimError(rc, "pansim_tree_newick failed")
    return buf.raw[:n.value].decode()


class NJTree(NamedTuple):
    """A neighbour-joining tree (pansim_nj_tree, include/pansim_b200.h): parent (uint32, root 0xFFFFFFFF) and the
    branch length above each node (float64, root 0) over n_leaves leaves, a node table the parsimony calls accept."""
    parent: np.ndarray
    length: np.ndarray
    n_leaves: int

    def newick(self) -> str:
        return tree_newick(self.parent, self.length, self.n_leaves)


class SplitComparison(NamedTuple):
    """pansim_tree_compare_splits: the non-trivial splits of each tree, those they share, and Robinson-Foulds
    rf = splits_a + splits_b - 2 shared."""
    splits_a: int
    splits_b: int
    shared: int
    rf: int


def compare_splits(a, b, n_leaves: int) -> SplitComparison:
    """The split comparison of two node tables over the same leaves (NJTree, Genealogy or parent arrays; no device)."""
    pa, pb = _parent_table(a), _parent_table(b)
    out = np.zeros(3, np.uint64)
    rc = _ffi.lib().pansim_tree_compare_splits(_ptr(pa), len(pa), _ptr(pb), len(pb), n_leaves, _ptr(out))
    if rc != OK:
        raise PansimError(rc, "pansim_tree_compare_splits: not node tables over that many leaves")
    sa, sb, sh = (int(x) for x in out)
    return SplitComparison(sa, sb, sh, sa + sb - 2 * sh)


def _nj_tree(call, check, n_leaves: int) -> NJTree:
    """call(parent, length) -> status."""
    parent = np.zeros(nj_nodes(n_leaves), np.uint32)
    length = np.zeros(len(parent), np.float64)
    check(call(_ptr(parent), _ptr(length)))
    return NJTree(parent, length, n_leaves)


def _genealogy(call, check, N: int) -> Genealogy:
    nodes = np.empty((2 * N, 3), np.uint32)
    info = _ffi.GenealogyInfo()
    check(call(_ptr(nodes), C.byref(info)))
    t = nodes[:info.n_nodes]
    return Genealogy(t[:, 0].copy(), t[:, 1].copy(), t[:, 2].copy(), info.generations_total, info.generations_kept,
                     info.n_nodes, info.lineages_at_start, N)


def _genealogy_history(lib, h, check, N: int) -> np.ndarray:
    info = _ffi.GenealogyInfo()
    check(lib.pansim_genealogy(h, None, C.byref(info)))
    out = np.empty((info.generations_kept, N), np.uint32)
    check(lib.pansim_genealogy_history(h, _ptr(out)))
    return out


def _tmrca(call, check, range1, range2) -> np.ndarray:
    r1 = np.ascontiguousarray(range1, np.uint32)
    r2 = np.ascontiguousarray(range2, np.uint32)
    assert r1.shape == r2.shape
    out = np.empty(len(r1), np.uint32)
    check(call(_ptr(r1), _ptr(r2), len(r1), _ptr(out)))
    return out


def _pairs_or_none(range1, range2):
    if range1 is None:
        return None, None, 0
    r1 = np.ascontiguousarray(range1, np.uint32)
    r2 = np.ascontiguousarray(range2, np.uint32)
    assert r1.shape == r2.shape
    return r1, r2, len(r1)


class Pansim:
    """Both populations of one run on one GPU (optionally one column shard of the core)."""

    def __init__(self, cfg: _ffi.Config):
        self._lib = _ffi.lib()
        self.cfg = cfg
        h = C.c_void_p()
        rc = self._lib.pansim_create(C.byref(cfg), C.byref(h))
        if rc != OK:
            raise PansimError(rc, self._lib.pansim_last_error(None).decode())
        self._h = h
        self.N, self.G, self.L = cfg.pop_size, cfg.pan_size, cfg.core_size
        info = self.info()
        self.local_sites = info.local_sites

    # -- lifecycle ---------------------------------------------------------
    @classmethod
    def from_params(cls, p: Params, device: int = 0, site_begin: int = 0, site_end: int = 0) -> "Pansim":
        return cls(make_config(p, device=device, site_begin=site_begin, site_end=site_end))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.pansim_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc: int):
        if rc != OK:
            raise PansimError(rc, self._lib.pansim_last_error(self._h).decode())

    def info(self) -> _ffi.Info:
        i = _ffi.Info()
        self._check(self._lib.pansim_get_info(self._h, C.byref(i)))
        return i

    def timing(self) -> _ffi.Timing:
        t = _ffi.Timing()
        self._check(self._lib.pansim_get_timing(self._h, C.byref(t)))
        return t

    def set_timing(self, enabled: bool):
        self._check(self._lib.pansim_set_timing(self._h, int(enabled)))

    def rates(self) -> np.ndarray:
        out = np.zeros(4, np.float64)
        self._check(self._lib.pansim_get_rates(self._h, _ptr(out)))
        return out

    # -- state -------------------------------------------------------------
    def set_initial(self, core_row_onehot, acc_row):
        """Population::new x2 (population.rs:199-230): every row = the given row."""
        cr = np.ascontiguousarray(core_row_onehot, np.uint8)
        ar = np.ascontiguousarray(acc_row, np.uint8)
        assert cr.shape == (self.L,) and ar.shape == (self.G,)
        self._check(self._lib.pansim_set_initial(self._h, _ptr(cr), _ptr(ar)))

    def upload(self, core_onehot=None, acc=None):
        if core_onehot is not None:
            c = np.ascontiguousarray(core_onehot, np.uint8)
            assert c.shape == (self.N, self.local_sites)
            self._check(self._lib.pansim_upload_core(self._h, _ptr(c)))
        if acc is not None:
            a = np.ascontiguousarray(acc, np.uint8)
            assert a.shape == (self.N, self.G)
            self._check(self._lib.pansim_upload_acc(self._h, _ptr(a)))

    def download_core(self) -> np.ndarray:
        out = np.empty((self.N, self.local_sites), np.uint8)
        self._check(self._lib.pansim_download_core(self._h, _ptr(out)))
        return out

    def download_acc(self) -> np.ndarray:
        out = np.empty((self.N, self.G), np.uint8)
        self._check(self._lib.pansim_download_acc(self._h, _ptr(out)))
        return out

    def export_core_csv(self, row_begin: int, row_end: int) -> bytes:
        out = np.empty((row_end - row_begin) * 2 * self.local_sites, np.uint8)
        self._check(self._lib.pansim_export_core_csv(self._h, row_begin, row_end, _ptr(out)))
        return out.tobytes()

    def set_selection(self, s):
        s = np.ascontiguousarray(s, np.float64)
        assert s.shape == (self.G,)
        self._check(self._lib.pansim_set_selection(self._h, _ptr(s)))

    # -- operators (names of population.rs) --------------------------------
    def average_distance(self) -> np.ndarray:
        """population.rs:753-784 on the accessory population."""
        out = np.empty(self.N, np.float64)
        self._check(self._lib.pansim_average_distance(self._h, _ptr(out)))
        return out

    def sample_indices(self, gen: int, avg_pairwise_dists=None) -> np.ndarray:
        """population.rs:270-448. Raises PansimError(PANSIM_ERR_WEIGHTS) where the
        reference's WeightedIndex::new(...).unwrap() panics."""
        avg = None if avg_pairwise_dists is None else np.ascontiguousarray(avg_pairwise_dists, np.float64)
        out = np.empty(self.N, np.uint32)
        self._check(self._lib.pansim_sample_indices(self._h, gen, _ptr(avg), _ptr(out)))
        return out

    def select_parents(self, gen: int, reuse: bool = False):
        """main.rs:435-443 in one call (one synchronisation): (avg_pairwise_dists, parents).
        reuse=True returns the object's own two arrays (overwritten by the next call) instead of fresh ones:
        a generation loop that only hands the parents on to step_with_parents saves the allocations."""
        if reuse:
            if not hasattr(self, "_sel_bufs"):
                a, o = np.empty(self.N, np.float64), np.empty(self.N, np.uint32)
                self._sel_bufs = (a, o, _ptr(a), _ptr(o))
            avg, out, pa, po = self._sel_bufs
        else:
            avg, out = np.empty(self.N, np.float64), np.empty(self.N, np.uint32)
            pa, po = _ptr(avg), _ptr(out)
        rc = self._lib.pansim_select_parents(self._h, gen, pa, po)
        if rc != OK:
            self._check(rc)
        return avg, out

    def weights(self):
        w = np.empty(self.N, np.float64)
        ng = np.empty(self.N, np.int32)
        lf = np.empty(self.N, np.float64)
        self._check(self._lib.pansim_get_weights(self._h, _ptr(w), _ptr(ng), _ptr(lf)))
        return w, ng, lf

    def next_generation(self, parents):
        """population.rs:450-465 for both populations (main.rs:445-447)."""
        p = np.ascontiguousarray(parents, np.uint32)
        assert p.shape == (self.N,)
        self._check(self._lib.pansim_next_generation(self._h, _ptr(p)))

    def step_with_parents(self, gen: int, parents):
        """main.rs:445-464 with host-supplied parents (generate mode)."""
        p = parents if (isinstance(parents, np.ndarray) and parents.dtype == np.uint32 and parents.flags.c_contiguous) \
            else np.ascontiguousarray(parents, np.uint32)
        assert p.shape == (self.N,)
        rc = self._lib.pansim_step_with_parents(self._h, gen, p.ctypes.data)
        if rc != OK:
            self._check(rc)

    def step(self, gen: int):
        """main.rs:435-464 entirely on the device."""
        self._check(self._lib.pansim_step(self._h, gen))

    def run_generations(self, gen0: int, n: int):
        self._check(self._lib.pansim_run_generations(self._h, gen0, n))

    def parents(self) -> np.ndarray:
        out = np.empty(self.N, np.uint32)
        self._check(self._lib.pansim_get_parents(self._h, _ptr(out)))
        return out

    def step_replay(self, parents, core_mut=None, acc_flip=None, hr=None, hgt=None):
        """Replay one generation from explicit events (apply order).
        core_mut = (row, site, allele_onehot); acc_flip = (row, gene);
        hr = (recipient, locus, value_onehot); hgt = (recipient, gene)."""
        keep = []

        def arr(x, dt):
            a = np.ascontiguousarray(x, dt)
            keep.append(a)
            return a

        e = _ffi.Events()
        e.parents = _ptr(arr(parents, np.uint32))
        if core_mut is not None and len(core_mut[0]):
            e.n_core_mut = len(core_mut[0])
            e.core_mut_row = _ptr(arr(core_mut[0], np.uint32))
            e.core_mut_site = _ptr(arr(core_mut[1], np.uint32))
            e.core_mut_allele = _ptr(arr(core_mut[2], np.uint8))
        if acc_flip is not None and len(acc_flip[0]):
            e.n_acc_flip = len(acc_flip[0])
            e.acc_flip_row = _ptr(arr(acc_flip[0], np.uint32))
            e.acc_flip_gene = _ptr(arr(acc_flip[1], np.uint32))
        if hr is not None and len(hr[0]):
            e.n_hr = len(hr[0])
            e.hr_recipient = _ptr(arr(hr[0], np.uint32))
            e.hr_locus = _ptr(arr(hr[1], np.uint32))
            e.hr_value = _ptr(arr(hr[2], np.uint8))
        if hgt is not None and len(hgt[0]):
            e.n_hgt = len(hgt[0])
            e.hgt_recipient = _ptr(arr(hgt[0], np.uint32))
            e.hgt_gene = _ptr(arr(hgt[1], np.uint32))
        self._check(self._lib.pansim_step_replay(self._h, C.byref(e)))

    # -- distances / reductions -------------------------------------------
    def pair_counts(self, range1, range2, core=True, acc=True):
        """Integer outputs of population.rs:787-837: (core_diff, inter, union)."""
        r1 = np.ascontiguousarray(range1, np.uint32)
        r2 = np.ascontiguousarray(range2, np.uint32)
        P = len(r1)
        cd = np.empty(P, np.uint32) if core else None
        it = np.empty(P, np.uint32) if acc else None
        un = np.empty(P, np.uint32) if acc else None
        self._check(self._lib.pansim_pair_counts(self._h, _ptr(r1), _ptr(r2), P, _ptr(cd), _ptr(it), _ptr(un)))
        return cd, it, un

    def pair_counts_device(self, range1, range2, d_core_diff: int, d_inter: int, d_uni: int):
        """Same, into caller-owned device buffers (raw pointers, e.g. tensor.data_ptr())."""
        r1 = np.ascontiguousarray(range1, np.uint32)
        r2 = np.ascontiguousarray(range2, np.uint32)
        self._check(self._lib.pansim_pair_counts_device(self._h, _ptr(r1), _ptr(r2), len(r1),
                                                        C.c_void_p(d_core_diff), C.c_void_p(d_inter),
                                                        C.c_void_p(d_uni)))

    def distances_from_counts(self, core_diff, inter, uni):
        """The f64 formulas of population.rs:822 and :828-830 (IEEE double ops,
        identical to pansim_core_distance / pansim_acc_distance)."""
        cg = float(self.cfg.core_genes)
        core_d = core_diff.astype(np.float64) / float(self.L)
        acc_d = 1.0 - ((inter.astype(np.float64) + cg) / (uni.astype(np.float64) + cg))
        return core_d, acc_d

    def pairwise_distances(self, range1, range2):
        """population.rs:787-837 for both populations -> (core_distances, acc_distances)."""
        cd, it, un = self.pair_counts(range1, range2)
        return self.distances_from_counts(cd, it, un)

    def pair_stats(self, range1, range2) -> tuple[float, float, float, float]:
        """main.rs:502-519 on the device: (avg_core, std_core, avg_acc, std_acc) of one distance pass,
        sums in the reference's left-to-right order (population.rs:87-94)."""
        r1 = np.ascontiguousarray(range1, np.uint32)
        r2 = np.ascontiguousarray(range2, np.uint32)
        out = np.empty(4, np.float64)
        self._check(self._lib.pansim_pair_stats(self._h, _ptr(r1), _ptr(r2), len(r1), _ptr(out)))
        return tuple(float(x) for x in out)

    def run_generations_stats(self, gen0: int, n: int, range1, range2) -> np.ndarray:
        """n generations, each followed by the distance pass and its statistics, in one device-resident
        batch (the --print_dist loop, main.rs:429-519): array [n, 4] of (avg_core, std_core, avg_acc, std_acc)."""
        r1 = np.ascontiguousarray(range1, np.uint32)
        r2 = np.ascontiguousarray(range2, np.uint32)
        out = np.empty((n, 4), np.float64)
        self._check(self._lib.pansim_run_generations_stats(self._h, gen0, n, _ptr(r1), _ptr(r2), len(r1), _ptr(out)))
        return out

    # -- core-genome diversity (extension) ---------------------------------
    def core_allele_counts(self) -> np.ndarray:
        """Per-site allele counts of the local sites: uint32 [local_sites, 4] = n_A, n_C, n_G, n_T."""
        out = np.empty((self.local_sites, 4), np.uint32)
        self._check(self._lib.pansim_core_allele_counts(self._h, _ptr(out)))
        return out

    def core_diversity(self, sfs: bool = False):
        """Diversity of the current core state; with sfs=True also (Diversity, sfs[N + 1] uint64), where sfs[k]
        counts the sites at which k individuals differ from the row given to set_initial."""
        d = _ffi.Diversity()
        h = np.empty(self.N + 1, np.uint64) if sfs else None
        self._check(self._lib.pansim_core_diversity(self._h, C.byref(d), _ptr(h)))
        return (_diversity(d), h) if sfs else _diversity(d)

    def run_generations_diversity(self, gen0: int, n: int, range1=None, range2=None):
        """n generations in one device-resident batch, each followed by the diversity reduction: (list of n
        Diversity, stats). With pairs, stats is the [n, 4] array of run_generations_stats (same bits); else None."""
        r1, r2, P = _pairs_or_none(range1, range2)
        divs = (_ffi.Diversity * max(n, 1))()
        st = np.empty((n, 4), np.float64) if P else None
        self._check(self._lib.pansim_run_generations_diversity(self._h, gen0, n, _ptr(r1), _ptr(r2), P, _ptr(st), divs))
        return [_diversity(divs[g]) for g in range(n)], st

    # -- core-genome linkage disequilibrium (extension) --------------------
    def core_ld(self, max_dist: int = 10000, bin_width: int = 100, min_minor: int = 1, next: "Pansim | None" = None) -> CoreLD:
        """r^2 and four-gamete pairs of the used sites binned by distance (pansim_core_ld). `next` is the context
        holding the sites right after this one's: its first max_dist sites are then the halo of this context, so the
        sum over the shards chained this way equals the single-context result."""
        bins, n = _ld_bins(max_dist, bin_width)
        used = C.c_uint64(0)
        self._check(self._lib.pansim_core_ld(self._h, next._h if next is not None else None,
                                             C.byref(_ld_params(max_dist, bin_width, min_minor)), bins, C.byref(used)))
        return _core_ld(bins, n, max_dist, bin_width, used.value)

    def ld_kernel_ms(self, max_dist: int = 10000, bin_width: int = 100, min_minor: int = 1, repeats: int = 10):
        """Measurement: device ms of one site pass, one transpose and one pair pass, and the pairs counted."""
        s, t, q, n = C.c_float(), C.c_float(), C.c_float(), C.c_uint64()
        self._check(self._lib.pansim_core_ld_kernel_ms(self._h, C.byref(_ld_params(max_dist, bin_width, min_minor)), repeats,
                                                       C.byref(s), C.byref(t), C.byref(q), C.byref(n)))
        return s.value, t.value, q.value, n.value

    # -- accessory-gene linkage (extension) ---------------------------------
    def gene_ld(self, r2_bins: int = 20, min_minor: int = 1) -> GeneLD:
        """r^2, associated, dissociated and four-gamete pairs of the used accessory genes by compartment class, and
        the r^2 histogram of each class (pansim_gene_ld)."""
        return _gene_ld(lambda *a: self._lib.pansim_gene_ld(self._h, *a), self._check, r2_bins, min_minor)

    def gene_ld_kernel_ms(self, r2_bins: int = 20, min_minor: int = 1, repeats: int = 10):
        """Measurement: device ms of one gene pass, one transpose and one pair pass, and the pairs counted."""
        g, t, q, n = C.c_float(), C.c_float(), C.c_float(), C.c_uint64()
        self._check(self._lib.pansim_gene_ld_kernel_ms(self._h, C.byref(_ffi.GeneLdParams(r2_bins, min_minor)), repeats,
                                                       C.byref(g), C.byref(t), C.byref(q), C.byref(n)))
        return g.value, t.value, q.value, n.value

    # -- pangenome accumulation (extension) ---------------------------------
    def gene_accumulation(self, n_perms: int = 100, seed: int | None = None) -> GeneAccumulation:
        """Pan, core, new and unique genes against the number of genomes over n_perms random orders of the rows,
        the orders drawn on the device from `seed` (None: the context's seed) (pansim_gene_accumulation)."""
        return _gene_accumulation(lambda *a: self._lib.pansim_gene_accumulation(self._h, *a), self._check, self.N, n_perms,
                                  self.cfg.seed if seed is None else seed)

    def gene_accumulation_kernel_ms(self, n_perms: int = 100, seed: int | None = None, repeats: int = 10):
        """Measurement: device ms of one order draw and of one accumulation, and the row bytes the walk reads."""
        o, a, n = C.c_float(), C.c_float(), C.c_uint64()
        self._check(self._lib.pansim_gene_accumulation_kernel_ms(self._h, self.cfg.seed if seed is None else seed, n_perms,
                                                                 repeats, C.byref(o), C.byref(a), C.byref(n)))
        return o.value, a.value, n.value

    def gene_spectrum(self) -> np.ndarray:
        """uint64 [N + 1]: the accessory genes carried by k rows, the core_genes added to bin N (pansim_gene_spectrum)."""
        return _gene_spectrum(lambda *a: self._lib.pansim_gene_spectrum(self._h, *a), self._check, self.N)

    # -- clonal genealogy (extension) ---------------------------------------
    def enable_genealogy(self, capacity: int):
        """Record the parent vector of every generation from now on, keeping the last `capacity` (0: stop and free)."""
        self._check(self._lib.pansim_enable_genealogy(self._h, capacity))

    def genealogy(self) -> Genealogy:
        """The genealogy of the present population traced on the device from the record."""
        return _genealogy(lambda nodes, info: self._lib.pansim_genealogy(self._h, nodes, info), self._check, self.N)

    def genealogy_history(self) -> np.ndarray:
        """The record itself: uint32 [kept, N], oldest generation first; row t maps child -> parent index."""
        return _genealogy_history(self._lib, self._h, self._check, self.N)

    def tmrca(self, range1, range2) -> np.ndarray:
        """Time to the most recent common ancestor of each pair (generations; the kept generations when the pair has
        not coalesced within the record)."""
        return _tmrca(lambda *a: self._lib.pansim_genealogy_tmrca(self._h, *a), self._check, range1, range2)

    # -- parsimony on the genealogy (extension) ------------------------------
    def core_parsimony(self, genealogy=None) -> CoreParsimony:
        """Parsimony changes of every local core site on a node table: a Genealogy, a parent array, or None for
        self.genealogy() (pansim_core_parsimony)."""
        parent = _parent_table(self.genealogy() if genealogy is None else genealogy)
        return _parsimony(lambda *a: self._lib.pansim_core_parsimony(self._h, *a), self._check, parent, self.local_sites, False)

    def gene_parsimony(self, genealogy=None) -> GeneParsimony:
        """Parsimony changes, gains and losses of every accessory gene on a node table (pansim_gene_parsimony)."""
        parent = _parent_table(self.genealogy() if genealogy is None else genealogy)
        return _parsimony(lambda *a: self._lib.pansim_gene_parsimony(self._h, *a), self._check, parent, self.G, True)

    def parsimony_kernel_ms(self, genealogy=None, genes: bool = False, repeats: int = 10):
        """Measurement: device ms of one parsimony pass (every slab), the bytes its walk reads, and the slabs."""
        parent = _parent_table(self.genealogy() if genealogy is None else genealogy)
        ms, nb, sl = C.c_float(), C.c_uint64(), C.c_uint32()
        self._check(self._lib.pansim_parsimony_kernel_ms(self._h, _ptr(parent), len(parent), int(genes), repeats,
                                                         C.byref(ms), C.byref(nb), C.byref(sl)))
        return ms.value, nb.value, sl.value

    # -- neighbour-joining (extension) -----------------------------------------
    def nj_tree(self, metric: str = "core") -> NJTree:
        """The neighbour-joining tree of the present rows on the core or accessory distances of <outpref>.tsv over
        every pair (pansim_nj_tree)."""
        m = NJ_METRICS[metric]
        return _nj_tree(lambda *a: self._lib.pansim_nj_tree(self._h, m, *a), self._check, self.N)

    def nj_tree_matrix(self, upper, n: int) -> NJTree:
        """The neighbour-joining tree of a caller's distances given as the upper triangle, row-major (n (n - 1) / 2
        values), on this context's device (pansim_nj_tree_matrix)."""
        upper = np.ascontiguousarray(upper, np.float64)
        if len(upper) != n * (n - 1) // 2:
            raise ValueError(f"{len(upper)} values for the upper triangle of {n} leaves")
        return _nj_tree(lambda *a: self._lib.pansim_nj_tree_matrix(self._h, _ptr(upper), n, *a), self._check, n)

    def nj_kernel_ms(self, metric: str = "core", repeats: int = 3):
        """Measurement: device ms of the matrix build and of the join loop, bytes the scans read, compactions."""
        b, j, nb, nc = C.c_float(), C.c_float(), C.c_uint64(), C.c_uint32()
        self._check(self._lib.pansim_nj_kernel_ms(self._h, NJ_METRICS[metric], repeats, C.byref(b), C.byref(j), C.byref(nb),
                                                  C.byref(nc)))
        return b.value, j.value, nb.value, nc.value

    # -- multi-GPU: communicator over column shards (one process per GPU) --
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = (C.c_uint8 * _ffi.COMM_ID_BYTES)()
        rc = _ffi.lib().pansim_comm_unique_id(C.byref(buf))
        if rc != OK:
            raise PansimError(rc, _ffi.lib().pansim_last_error(None).decode())
        return bytes(buf)

    def comm_init_rank(self, n_ranks: int, rank: int, unique_id: bytes):
        """ncclCommInitRank inside the library: from now on the pair-count calls return
        whole-alignment core counts (summed over the column shards on the device)."""
        assert len(unique_id) == _ffi.COMM_ID_BYTES
        buf = (C.c_uint8 * _ffi.COMM_ID_BYTES).from_buffer_copy(unique_id)
        self._check(self._lib.pansim_comm_init_rank(self._h, n_ranks, rank, C.byref(buf)))

    def pairs_in_rows(self, row_begin: int, row_end: int) -> int:
        """Number of pairs (i, j) with row_begin <= i < row_end, i < j < N."""
        n = row_end - row_begin
        return n * (self.N - 1) - (row_begin + row_end - 1) * n // 2

    def pair_counts_rows(self, row_begin: int, row_end: int, core: bool = True, acc: bool = True):
        """Exact all-pairs mode for one block of rows (extension; the reference only samples pairs
        with replacement, main.rs:413-427): (core_diff, inter, union) of every pair (i, j),
        row_begin <= i < row_end, i < j < N, ordered by i then j. The pair list is generated on
        the device."""
        P = self.pairs_in_rows(row_begin, row_end)
        cd = np.empty(P, np.uint32) if core else None
        it = np.empty(P, np.uint32) if acc else None
        un = np.empty(P, np.uint32) if acc else None
        n = C.c_size_t(0)
        self._check(self._lib.pansim_pair_counts_rows(self._h, row_begin, row_end, _ptr(cd), _ptr(it), _ptr(un),
                                                      C.byref(n)))
        assert n.value == P
        return cd, it, un

    def pair_counts_rows_device(self, row_begin: int, row_end: int, d_core_diff: int, d_inter: int, d_uni: int) -> int:
        """Same, into caller-owned device buffers (raw pointers); returns the number of pairs."""
        n = C.c_size_t(0)
        self._check(self._lib.pansim_pair_counts_rows_device(self._h, row_begin, row_end, C.c_void_p(d_core_diff),
                                                             C.c_void_p(d_inter), C.c_void_p(d_uni), C.byref(n)))
        return n.value

    def row_blocks(self, chunk_pairs: int = 4_000_000):
        """Row blocks [i0, i1) of about `chunk_pairs` pairs each covering every i < N - 1."""
        N, i0 = self.N, 0
        while i0 < N - 1:
            i1, n = i0, 0
            while i1 < N - 1 and (n == 0 or n + (N - 1 - i1) <= chunk_pairs):
                n += N - 1 - i1
                i1 += 1
            yield i0, i1
            i0 = i1

    def iter_all_pairs(self, chunk_pairs: int = 4_000_000, with_indices: bool = True):
        """Exact all-pairs mode: yields (i, j, core_diff, inter, union) arrays covering every
        unordered pair i < j exactly once, in chunks of about `chunk_pairs` pairs (i, j are None
        with with_indices=False: the order is i ascending, then j ascending)."""
        N = self.N
        for i0, i1 in self.row_blocks(chunk_pairs):
            cd, it, un = self.pair_counts_rows(i0, i1)
            ii = jj = None
            if with_indices:
                ii = np.repeat(np.arange(i0, i1, dtype=np.uint32), [N - 1 - i for i in range(i0, i1)])
                jj = np.concatenate([np.arange(i + 1, N, dtype=np.uint32) for i in range(i0, i1)])
            yield ii, jj, cd, it, un

    def gene_counts(self) -> np.ndarray:
        out = np.empty(self.G, np.uint32)
        self._check(self._lib.pansim_gene_counts(self._h, _ptr(out)))
        return out

    def gene_frequencies(self) -> np.ndarray:
        """population.rs:840-863: accessory frequencies then core_genes x 1.0."""
        f = self.gene_counts().astype(np.float64) / float(self.N)
        return np.concatenate([f, np.ones(self.cfg.core_genes, np.float64)])

    def calc_gene_freq(self) -> float:
        """population.rs:244-268: mean over rows of (row sum / G), sequential sums."""
        acc = self.download_acc()
        props = acc.sum(axis=1).astype(np.float64) / float(self.G)
        return float(np.cumsum(props)[-1]) / float(self.N)

    # -- instrumentation ---------------------------------------------------
    def enable_event_dump(self, max_core_events: int):
        self._check(self._lib.pansim_enable_event_dump(self._h, max_core_events))

    def fetch_event_dump(self) -> dict:
        d = _ffi.EventDump()
        self._check(self._lib.pansim_fetch_event_dump(self._h, C.byref(d)))

        def cp(ptr, n, dt):
            return np.ctypeslib.as_array(ptr, shape=(n,)).astype(dt, copy=True) if n else np.zeros(0, dt)

        out = dict(
            core_mut_row=cp(d.core_mut_row, d.n_core_mut, np.uint32),
            core_mut_site=cp(d.core_mut_site, d.n_core_mut, np.uint32),
            core_mut_seq=cp(d.core_mut_seq, d.n_core_mut, np.uint32),
            core_mut_allele=cp(d.core_mut_allele, d.n_core_mut, np.uint8),
            hr_recipient=cp(d.hr_recipient, d.n_hr, np.uint32),
            hr_locus=cp(d.hr_locus, d.n_hr, np.uint32),
            hr_donor=cp(d.hr_donor, d.n_hr, np.uint32),
            hr_seq=cp(d.hr_seq, d.n_hr, np.uint32),
            hr_value=cp(d.hr_value, d.n_hr, np.uint8),
            acc_flip_mask=cp(d.acc_flip_mask, self.N * self.G, np.uint8).reshape(self.N, self.G),
            acc_gain_mask=cp(d.acc_gain_mask, self.N * self.G, np.uint8).reshape(self.N, self.G),
        )
        self._lib.pansim_free_event_dump(C.byref(d))
        return out

    # -- writers (population.rs:865-897) ------------------------------------
    def write_core_csv(self, path: str) -> int:
        """_core_genome.csv written by the library (GPU text expansion, pinned double-buffered streaming); bytes written."""
        n = C.c_uint64(0)
        self._check(self._lib.pansim_write_core_csv(self._h, path.encode(), C.byref(n)))
        return n.value

    def write_core_vcf(self, path: str, header: bool = True) -> int:
        """The core alignment as VCF 4.2 (include/pansim_b200.h): one line per site where some row differs from
        the row given to set_initial, haploid GT against it. A column-shard context writes its own lines with
        global POS; header=False leaves out the header, so the shards' bodies can be concatenated. Bytes written."""
        n = C.c_uint64(0)
        self._check(self._lib.pansim_write_core_vcf(self._h, path.encode(), int(header), C.byref(n)))
        return n.value

    def vcf_kernel_ms(self, repeats: int = 10) -> tuple[float, float, int]:
        """Measurement: device ms of one VCF site pass and of one expansion of every chunk (no copy), and the
        bytes of text (header excluded)."""
        site, expand, n = C.c_float(), C.c_float(), C.c_uint64()
        self._check(self._lib.pansim_core_vcf_kernel_ms(self._h, repeats, C.byref(site), C.byref(expand), C.byref(n)))
        return site.value, expand.value, n.value

    def write_core_fasta(self, path: str, snps_only: bool = False) -> CoreFasta:
        """The core alignment as FASTA (include/pansim_b200.h): one record `>ind_<i>` per row, every site as a column
        or, with snps_only, the sites where two or more letters are present (snp-sites' selection). Returns the
        bytes written, the columns and the constant-site counts by letter (A, C, G, T)."""
        return _write_fasta(lambda *a: self._lib.pansim_write_core_fasta(self._h, *a), self._check, path, snps_only)

    def export_core_fasta_rows(self, row_begin: int, row_end: int, snps_only: bool = False) -> np.ndarray:
        """The FASTA letters of rows [row_begin, row_end) without headers: uint8 [rows, columns] of ASCII ACGT. On a
        column shard the columns are the shard's own; the shards' arrays, concatenated along axis 1 in shard order,
        are the whole alignment's. In whole mode the columns are the local sites; in SNP mode a first call (out = NULL)
        asks for their number, which repeats the site pass of the second (0.1-0.6 ms on a B200 at 1 000 to
        10 000 x 1.2 Mbp, profiles/r07_fasta_bench.json)."""
        cols = C.c_uint64(self.local_sites)
        if snps_only:
            self._check(self._lib.pansim_export_core_fasta_rows(self._h, 1, row_begin, row_end, None, C.byref(cols)))
        out = np.empty((max(0, row_end - row_begin), cols.value), np.uint8)
        self._check(self._lib.pansim_export_core_fasta_rows(self._h, int(snps_only), row_begin, row_end, _ptr(out),
                                                            C.byref(cols)))
        return out

    def fasta_kernel_ms(self, snps_only: bool = False, repeats: int = 10) -> tuple[float, float, int]:
        """Measurement: device ms of one FASTA site pass (SNP mode) and of one expansion of every chunk of records
        (no copy), and the bytes of the file."""
        site, expand, n = C.c_float(), C.c_float(), C.c_uint64()
        self._check(self._lib.pansim_core_fasta_kernel_ms(self._h, int(snps_only), repeats, C.byref(site), C.byref(expand),
                                                          C.byref(n)))
        return site.value, expand.value, n.value

    def write(self, outpref: str):
        self.write_core_csv(outpref + "_core_genome.csv")
        acc = self.download_acc()
        with open(outpref + "_pangenome.csv", "w") as f:
            ones = ["1"] * self.cfg.core_genes                                   # :891
            for r in range(self.N):
                f.write(",".join(ones + [str(int(x)) for x in acc[r]]) + "\n")


__all__ = ["Pansim", "PansimError", "Diversity", "diversity_stats", "CoreLD", "ld_mean_r2", "GeneLD", "GeneAccumulation",
           "pangenome_classes", "CoreParsimony", "GeneParsimony", "parsimony_indices", "NJTree", "SplitComparison",
           "compare_splits", "tree_newick", "Genealogy", "genealogy_newick",
           "make_config", "standard_deviation", "fmt_f64"]
