"""numpy reference of the pangenome accumulation curves, the gene frequency spectrum and Roary's gene classes
(include/pansim_b200.h, pansim_gene_accumulation / pansim_gene_spectrum / pansim_pangenome_classes), shared by the
gene-accumulation tests and tools/gene_accumulation_bench.py."""
import numpy as np

ORDER_TAG = 0x00A00000                       # PANSIM_GENE_ACC_ORDER_TAG
_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_LO = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Philox4x32-10 of common.cuh on arrays: ctr = four uint32 arrays (broadcast together), key = (k0, k1).
    Returns the four output words as uint32 arrays."""
    c = [np.asarray(x, np.uint64) & _LO for x in np.broadcast_arrays(*ctr)]
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    for _ in range(10):
        p0 = _M0 * c[0]                       # 32 x 32 bits: exact in uint64
        p1 = _M1 * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ np.uint64(k0), p1 & _LO, (p0 >> np.uint64(32)) ^ c[3] ^ np.uint64(k1), p0 & _LO]
        k0 = (k0 + _W0) & 0xFFFFFFFF
        k1 = (k1 + _W1) & 0xFFFFFFFF
    return tuple(x.astype(np.uint32) for x in c)


def np_orders(seed, n_perms, N):
    """uint32 [n_perms, N]: order p by Fisher-Yates from the identity, for i = N-1 down to 1 swapping o[i] and
    o[j], j = (r * (i + 1)) >> 32, r = .x of Philox4x32-10 with key (lo32(seed), hi32(seed)) and counter
    {i, p, 0, ORDER_TAG}."""
    P = int(n_perms)
    o = np.tile(np.arange(N, dtype=np.int64), (P, 1))
    if N < 2:
        return o.astype(np.uint32)
    i = np.arange(N, dtype=np.uint64)[None, :]
    p = np.arange(P, dtype=np.uint64)[:, None]
    r = philox4x32_10((i, p, 0, ORDER_TAG), (seed & 0xFFFFFFFF, seed >> 32))[0].astype(np.uint64)
    J = ((r * (i + np.uint64(1))) >> np.uint64(32)).astype(np.int64)
    rows = np.arange(P)
    for k in range(N - 1, 0, -1):
        j = J[:, k]
        t = o[:, k].copy()
        o[:, k] = o[rows, j]
        o[rows, j] = t
    return o.astype(np.uint32)


def np_curves(pres, orders, c0):
    """Per order p and k = 1..N, from cnt = cumsum(pres[order], axis=0): pan = (cnt > 0).sum + c0, core =
    (cnt == k).sum + c0, unique = (cnt == 1).sum (+ c0 at k = 1), new = diff(pan) with pan(0) = 0. Returns the four
    uint32 [P, N] arrays (pan, core, new, unique)."""
    pres = np.asarray(pres, bool)
    N = pres.shape[0]
    orders = np.asarray(orders, np.int64).reshape(-1, N)
    dt = np.int16 if N < 2 ** 15 else np.int32
    k = np.arange(1, N + 1, dtype=dt)[:, None]
    out = [np.zeros(orders.shape, np.int64) for _ in range(4)]
    for p, order in enumerate(orders):
        cnt = np.cumsum(pres[order], axis=0, dtype=dt)
        pan = (cnt > 0).sum(axis=1) + c0
        out[0][p] = pan
        out[1][p] = (cnt == k).sum(axis=1) + c0
        out[2][p] = np.diff(pan, prepend=0)
        out[3][p] = (cnt == 1).sum(axis=1)
        out[3][p, 0] += c0
    return tuple(x.astype(np.uint32) for x in out)


def np_spectrum(pres, c0):
    """uint64 [N + 1]: bincount of the presence counts a_g, + c0 in bin N."""
    pres = np.asarray(pres, bool)
    N = pres.shape[0]
    s = np.bincount(pres.sum(axis=0), minlength=N + 1).astype(np.uint64)
    s[N] += np.uint64(c0)
    return s


def np_classes(spectrum, N):
    """(core, soft core, shell, cloud, total) by Roary's thresholds as integer tests on a >= 1 rows."""
    out = [0] * 4
    for a in range(1, N + 1):
        h = 100 * a
        out[0 if h >= 99 * N else 1 if h >= 95 * N else 2 if h >= 15 * N else 3] += int(spectrum[a])
    return (*out, sum(out))
