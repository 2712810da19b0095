"""Several GPUs in one process: `PansimGroup` over the pansim_group_* C ABI.

The reference is one process whose Population methods are called from the main thread
(main.rs:429-528); this mirror keeps that shape and lets the library shard the core
alignment by columns over the devices of the box (NCCL inside the library, see
include/pansim_b200.h "multi-GPU"). Method names follow `Pansim`.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _ffi
from .params import Params
from .population import (NJ_METRICS, OK, CoreFasta, CoreLD, CoreParsimony, GeneAccumulation, GeneLD, GeneParsimony, Genealogy,
                         NJTree, PansimError, _core_ld, _diversity, _gene_accumulation, _gene_ld, _gene_spectrum, _genealogy, _genealogy_history,
                         _ld_bins, _ld_params, _nj_tree, _pairs_or_none, _parent_table, _parsimony, _ptr, _tmrca, _write_fasta,
                         make_config)


class PansimGroup:
    def __init__(self, p: Params, n_devices: int, devices=None):
        self._lib = _ffi.lib()
        self.cfg = make_config(p)
        devs = None
        if devices is not None:
            devs = (C.c_int * n_devices)(*devices)
        h = C.c_void_p()
        rc = self._lib.pansim_group_create(C.byref(self.cfg), n_devices, devs, C.byref(h))
        if rc != OK:
            raise PansimError(rc, self._lib.pansim_group_last_error(None).decode())
        self._h = h
        self.N, self.G, self.L = self.cfg.pop_size, self.cfg.pan_size, self.cfg.core_size
        self.size = self._lib.pansim_group_size(h)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.pansim_group_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != OK:
            raise PansimError(rc, self._lib.pansim_group_last_error(self._h).decode())

    def set_initial(self, core_row_onehot, acc_row):
        cr = np.ascontiguousarray(core_row_onehot, np.uint8)
        ar = np.ascontiguousarray(acc_row, np.uint8)
        assert cr.shape == (self.L,) and ar.shape == (self.G,)
        self._check(self._lib.pansim_group_set_initial(self._h, _ptr(cr), _ptr(ar)))

    def set_selection(self, s):
        s = np.ascontiguousarray(s, np.float64)
        self._check(self._lib.pansim_group_set_selection(self._h, _ptr(s)))

    def run_generations(self, gen0: int, n: int):
        self._check(self._lib.pansim_group_run_generations(self._h, gen0, n))

    def pair_counts(self, range1, range2):
        r1 = np.ascontiguousarray(range1, np.uint32)
        r2 = np.ascontiguousarray(range2, np.uint32)
        P = len(r1)
        cd, it, un = (np.empty(P, np.uint32) for _ in range(3))
        self._check(self._lib.pansim_group_pair_counts(self._h, _ptr(r1), _ptr(r2), P, _ptr(cd), _ptr(it), _ptr(un)))
        return cd, it, un

    def run_generations_stats(self, gen0: int, n: int, range1, range2) -> np.ndarray:
        r1 = np.ascontiguousarray(range1, np.uint32)
        r2 = np.ascontiguousarray(range2, np.uint32)
        out = np.empty((n, 4), np.float64)
        self._check(self._lib.pansim_group_run_generations_stats(self._h, gen0, n, _ptr(r1), _ptr(r2), len(r1), _ptr(out)))
        return out

    def all_pairs(self, chunk_pairs: int = 4_000_000):
        """Exact all-pairs mode: (core_diff, inter, union) of every pair i < j in (i, j) order."""
        parts = []

        def cb(_user, i0, i1, n, cd, it, un):
            parts.append((i0, i1, np.ctypeslib.as_array(cd, (n,)).copy(), np.ctypeslib.as_array(it, (n,)).copy(),
                          np.ctypeslib.as_array(un, (n,)).copy()))
            return 0

        self._check(self._lib.pansim_group_all_pairs(self._h, chunk_pairs, _ffi.PAIRS_CB(cb), None))
        return parts

    def walk_all_pairs(self, chunk_pairs: int = 4_000_000, sink=None) -> dict:
        """The same walk without keeping the vectors: `sink(i0, i1, core_diff, inter, union)` per block (views,
        valid during the call) or nothing. Returns wall ms, reduce-scatter device ms on shard 0, pairs."""
        def cb(_user, i0, i1, n, cd, it, un):
            if sink is not None:
                sink(i0, i1, np.ctypeslib.as_array(cd, (n,)), np.ctypeslib.as_array(it, (n,)), np.ctypeslib.as_array(un, (n,)))
            return 0

        self._check(self._lib.pansim_group_all_pairs(self._h, chunk_pairs, _ffi.PAIRS_CB(cb), None))
        wall, nccl, pairs = C.c_float(), C.c_float(), C.c_uint64()
        self._check(self._lib.pansim_group_all_pairs_timing(self._h, C.byref(wall), C.byref(nccl), C.byref(pairs)))
        return dict(wall_ms=wall.value, nccl_ms_shard0=nccl.value, pairs=pairs.value)

    def core_diversity(self, sfs: bool = False):
        """Whole-alignment diversity (shard partials summed); with sfs=True also the SFS [N + 1] (Pansim.core_diversity)."""
        d = _ffi.Diversity()
        h = np.empty(self.N + 1, np.uint64) if sfs else None
        self._check(self._lib.pansim_group_core_diversity(self._h, C.byref(d), _ptr(h)))
        return (_diversity(d), h) if sfs else _diversity(d)

    def core_allele_counts(self) -> np.ndarray:
        """uint32 [core_size, 4] assembled from the shards (Pansim.core_allele_counts per shard context)."""
        out = np.empty((self.L, 4), np.uint32)
        for i in range(self.size):
            h = self._lib.pansim_group_ctx(self._h, i)
            info = _ffi.Info()
            self._check(self._lib.pansim_get_info(h, C.byref(info)))
            part = np.empty((info.local_sites, 4), np.uint32)
            rc = self._lib.pansim_core_allele_counts(h, _ptr(part))
            if rc != OK:
                raise PansimError(rc, self._lib.pansim_last_error(h).decode())
            begin = self._shard_begin(i)
            out[begin:begin + info.local_sites] = part
        return out

    def _shard_begin(self, i: int) -> int:
        b, e = C.c_uint64(), C.c_uint64()
        self._check(self._lib.pansim_shard_bounds(self.L, self.size, i, C.byref(b), C.byref(e)))
        return b.value

    def run_generations_diversity(self, gen0: int, n: int, range1=None, range2=None):
        """Pansim.run_generations_diversity over the shards: (list of n whole-alignment Diversity, stats or None)."""
        r1, r2, P = _pairs_or_none(range1, range2)
        divs = (_ffi.Diversity * max(n, 1))()
        st = np.empty((n, 4), np.float64) if P else None
        self._check(self._lib.pansim_group_run_generations_diversity(self._h, gen0, n, _ptr(r1), _ptr(r2), P, _ptr(st), divs))
        return [_diversity(divs[g]) for g in range(n)], st

    def core_ld(self, max_dist: int = 10000, bin_width: int = 100, min_minor: int = 1) -> CoreLD:
        """Whole-alignment LD bins (Pansim.core_ld): every shard with the next one as its halo, summed."""
        bins, n = _ld_bins(max_dist, bin_width)
        used = C.c_uint64(0)
        self._check(self._lib.pansim_group_core_ld(self._h, C.byref(_ld_params(max_dist, bin_width, min_minor)), bins,
                                                   C.byref(used)))
        return _core_ld(bins, n, max_dist, bin_width, used.value)

    def gene_ld(self, r2_bins: int = 20, min_minor: int = 1) -> GeneLD:
        """Accessory-gene linkage (Pansim.gene_ld): the accessory matrix is replicated, so shard 0 answers."""
        return _gene_ld(lambda *a: self._lib.pansim_group_gene_ld(self._h, *a), self._check, r2_bins, min_minor)

    def gene_accumulation(self, n_perms: int = 100, seed: int | None = None) -> GeneAccumulation:
        """Pangenome accumulation curves (Pansim.gene_accumulation): the accessory matrix is replicated, so shard 0
        answers."""
        return _gene_accumulation(lambda *a: self._lib.pansim_group_gene_accumulation(self._h, *a), self._check, self.N,
                                  n_perms, self.cfg.seed if seed is None else seed)

    def gene_spectrum(self) -> np.ndarray:
        """The gene frequency spectrum (Pansim.gene_spectrum), answered by shard 0."""
        return _gene_spectrum(lambda *a: self._lib.pansim_group_gene_spectrum(self._h, *a), self._check, self.N)

    def core_parsimony(self, genealogy=None) -> CoreParsimony:
        """Pansim.core_parsimony over the whole alignment: every shard scores its sites, the results are summed and the
        site scores concatenated in site order."""
        parent = _parent_table(self.genealogy() if genealogy is None else genealogy)
        return _parsimony(lambda *a: self._lib.pansim_group_core_parsimony(self._h, *a), self._check, parent, self.L, False)

    def gene_parsimony(self, genealogy=None) -> GeneParsimony:
        """Pansim.gene_parsimony: the accessory matrix is replicated, so shard 0 answers."""
        parent = _parent_table(self.genealogy() if genealogy is None else genealogy)
        return _parsimony(lambda *a: self._lib.pansim_group_gene_parsimony(self._h, *a), self._check, parent, self.G, True)

    def nj_tree(self, metric: str = "core") -> NJTree:
        """Pansim.nj_tree of the group: core counts summed over the shards, shard 0 joins; the same tree as one
        context."""
        m = NJ_METRICS[metric]
        return _nj_tree(lambda *a: self._lib.pansim_group_nj_tree(self._h, m, *a), self._check, self.N)

    def enable_genealogy(self, capacity: int):
        """Pansim.enable_genealogy for the group: shard 0 records (every shard draws the same parents)."""
        self._check(self._lib.pansim_group_enable_genealogy(self._h, capacity))

    def genealogy(self) -> Genealogy:
        return _genealogy(lambda nodes, info: self._lib.pansim_group_genealogy(self._h, nodes, info), self._check, self.N)

    def genealogy_history(self) -> np.ndarray:
        h = self._lib.pansim_group_ctx(self._h, 0)

        def check(rc):
            if rc != OK:
                raise PansimError(rc, self._lib.pansim_last_error(h).decode())
        return _genealogy_history(self._lib, h, check, self.N)

    def tmrca(self, range1, range2) -> np.ndarray:
        return _tmrca(lambda *a: self._lib.pansim_group_genealogy_tmrca(self._h, *a), self._check, range1, range2)

    def gene_counts(self) -> np.ndarray:
        out = np.empty(self.G, np.uint32)
        self._check(self._lib.pansim_group_gene_counts(self._h, _ptr(out)))
        return out

    def download_acc(self) -> np.ndarray:
        out = np.empty((self.N, self.G), np.uint8)
        self._check(self._lib.pansim_group_download_acc(self._h, _ptr(out)))
        return out

    def download_core(self) -> np.ndarray:
        out = np.empty((self.N, self.L), np.uint8)
        self._check(self._lib.pansim_group_download_core(self._h, _ptr(out)))
        return out

    def write_core_vcf(self, path: str) -> int:
        """The whole-alignment VCF (Pansim.write_core_vcf): header once, then every shard's lines; bytes written."""
        n = C.c_uint64(0)
        self._check(self._lib.pansim_group_write_core_vcf(self._h, path.encode(), C.byref(n)))
        return n.value

    def write_core_fasta(self, path: str, snps_only: bool = False) -> CoreFasta:
        """The whole-alignment FASTA (Pansim.write_core_fasta): the shards' letters of every row in shard order; the
        columns and constant-site counts are summed over the shards."""
        return _write_fasta(lambda *a: self._lib.pansim_group_write_core_fasta(self._h, *a), self._check, path, snps_only)

    def export_core_csv(self, row_begin: int, row_end: int) -> bytes:
        out = np.empty((row_end - row_begin) * 2 * self.L, np.uint8)
        self._check(self._lib.pansim_group_export_core_csv(self._h, row_begin, row_end, _ptr(out)))
        return out.tobytes()
