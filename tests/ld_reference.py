"""numpy reference of the core-genome LD bins (include/pansim_b200.h, pansim_core_ld), shared by the LD tests."""
import numpy as np


def np_ld_from_derived(der, max_dist, bin_width, min_minor, site_begin=0):
    """Reference of include/pansim_b200.h from the derived matrix der [N, sites] (bool): per bin (pairs, four_gamete,
    sum of q as a Python int), and the used sites. float64 operations in the header's order, np.rint = round-half-even."""
    n = der.shape[0]
    a_all = der.sum(axis=0).astype(np.int64)
    used = np.flatnonzero(min_minor <= np.minimum(a_all, n - a_all))
    pos = used.astype(np.int64) + site_begin
    a = a_all[used]
    inv = 1.0 / (a * (n - a)).astype(np.float64)
    xf = der[:, used].astype(np.float32)                     # exact: counts <= n < 2^24
    nb = -(-max_dist // bin_width)
    pairs = np.zeros(nb, np.int64)
    fg = np.zeros(nb, np.int64)
    r2 = [0] * nb
    U, B = len(used), 1024
    for i0 in range(0, U, B):
        i1 = min(U, i0 + B)
        j1 = int(np.searchsorted(pos, pos[i1 - 1] + max_dist, side="right"))
        if j1 <= i0 + 1:
            continue
        c = np.rint(xf[:, i0:i1].T @ xf[:, i0:j1]).astype(np.int64)
        I, J = np.meshgrid(np.arange(i0, i1), np.arange(i0, j1), indexing="ij")
        d = pos[J] - pos[I]
        m = (J > I) & (d <= max_dist)
        c, I, J, d = c[m], I[m], J[m], d[m]
        if not len(d):
            continue
        ai, aj = a[I], a[J]
        D = (n * c - ai * aj).astype(np.float64)
        q = np.rint(((D * D) * inv[I]) * inv[J] * 2.0 ** 32).astype(np.uint64)
        four = (c > 0) & (ai - c > 0) & (aj - c > 0) & (n - ai - aj + c > 0)
        b = (d - 1) // bin_width
        pairs += np.bincount(b, minlength=nb)
        fg += np.bincount(b[four], minlength=nb)
        o = np.argsort(b, kind="stable")
        bs, qs = b[o], q[o]
        starts = np.flatnonzero(np.r_[True, bs[1:] != bs[:-1]])
        for k, s in zip(bs[starts], np.add.reduceat(qs, starts)):
            r2[int(k)] += int(s)
    return pairs, fg, r2, len(used)
