"""numpy reference of the accessory-gene linkage (include/pansim_b200.h, pansim_gene_ld), shared by the gene-LD tests."""
import numpy as np

CLASSES = ("0-0", "0-1", "1-1")


def gene_groups(G, n_compartments, comp_lo, comp_hi):
    """group(g) of the header: 1 for the genes of compartment 1 when there are two compartments, else 0."""
    grp = np.zeros(G, np.int64)
    if n_compartments == 2:
        grp[comp_lo[1]:comp_hi[1]] = 1
    return grp


def np_gene_ld(pres, grp, r2_bins, min_minor):
    """Reference of include/pansim_b200.h from the presence matrix pres [N, G] (bool) and the group of every gene.
    Returns a dict: per class (0-0, 0-1, 1-1) pairs, four_gamete, associated, dissociated, r2_sum (Python ints);
    hist [3, r2_bins] and genes_used [2]. c = X^T X exactly (float32 over 0/1 values below 2^24 rows, else int64);
    float64 operations in the header's order, np.rint = round-half-even."""
    pres = np.asarray(pres, bool)
    n, G = pres.shape
    grp = np.asarray(grp, np.int64)
    a_all = pres.sum(axis=0).astype(np.int64)
    used = np.flatnonzero(min_minor <= np.minimum(a_all, n - a_all)) if n >= 2 else np.zeros(0, np.int64)
    a = a_all[used]
    g = grp[used]
    inv = 1.0 / (a * (n - a)).astype(np.float64)
    x = pres[:, used].astype(np.float32 if n < 2 ** 24 else np.int64)
    out = dict(pairs=[0] * 3, four_gamete=[0] * 3, associated=[0] * 3, dissociated=[0] * 3, r2_sum=[0] * 3,
               hist=np.zeros((3, r2_bins), np.int64),
               genes_used=np.array([int((g == 0).sum()), int((g == 1).sum())], np.int64))
    U, B = len(used), 1024
    for i0 in range(0, U, B):
        i1 = min(U, i0 + B)
        c = np.rint(x[:, i0:i1].T @ x[:, i0:]).astype(np.int64) if x.dtype == np.float32 else x[:, i0:i1].T @ x[:, i0:]
        I, J = np.meshgrid(np.arange(i0, i1), np.arange(i0, U), indexing="ij")
        m = J > I
        c, I, J = c[m], I[m], J[m]
        if not len(c):
            continue
        ai, aj = a[I], a[J]
        D = n * c - ai * aj
        Df = D.astype(np.float64)
        q = np.rint(((Df * Df) * inv[I]) * inv[J] * 2.0 ** 32).astype(np.uint64)
        four = (c > 0) & (ai - c > 0) & (aj - c > 0) & (n - ai - aj + c > 0)
        cls = g[I] + g[J]
        b = np.minimum((q * np.uint64(r2_bins)) >> np.uint64(32), np.uint64(r2_bins - 1)).astype(np.int64)
        out["hist"] += np.bincount(cls * r2_bins + b, minlength=3 * r2_bins).reshape(3, r2_bins)
        for k in range(3):
            s = cls == k
            out["pairs"][k] += int(s.sum())
            out["four_gamete"][k] += int((four & s).sum())
            out["associated"][k] += int(((D > 0) & s).sum())
            out["dissociated"][k] += int(((D < 0) & s).sum())
            out["r2_sum"][k] += sum(int(v) for v in np.add.reduceat(q[s], np.arange(0, int(s.sum()), 1 << 20))) if s.any() else 0
    return out
