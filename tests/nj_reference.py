"""Numpy float64 reference of neighbour-joining as include/pansim_b200.h defines it (every operation in the stated
order, so it reproduces the device bit for bit), the distance matrices of the core and accessory metrics from
downloaded states, a pure-Python split comparison from leaf sets, a Newick writer, and additive tree metrics."""
import numpy as np

NONE = 0xFFFFFFFF


def nj_nodes(n):
    return 2 * n - 2 if n >= 3 else 3 if n == 2 else 1


def nj(D):
    """(parent uint32, length float64) of the tree of a full symmetric float64 matrix with a zero diagonal."""
    D = np.array(D, np.float64)
    n = len(D)
    parent = np.full(nj_nodes(n), NONE, np.uint32)
    length = np.zeros(nj_nodes(n), np.float64)
    if n == 1:
        return parent, length
    if n == 2:
        parent[:2] = 2
        length[:2] = D[0, 1] * 0.5
        return parent, length
    R = np.add.accumulate(D, axis=1)[:, -1].copy()           # left to right over ascending b
    active = list(range(n))                                  # matrix rows of the slots, in slot order
    node = list(range(n))                                    # node of each matrix row
    for t in range(n - 3):
        k = n - t
        idx = np.array(active)
        Q = ((k - 2) * D[np.ix_(idx, idx)] - R[idx][:, None]) - R[idx][None, :]
        Q[np.tril_indices(k)] = np.inf
        a, b = divmod(int(np.argmin(Q)), k)                  # first minimum in row-major order: smaller a, then b
        A, B = active[a], active[b]
        dab, ra, rb = D[A, B], R[A], R[B]
        da = (dab + (ra - rb) / (k - 2)) * 0.5
        db = dab - da
        u = n + t
        parent[node[A]], length[node[A]] = u, da
        parent[node[B]], length[node[B]] = u, db
        C = np.array([c for c in active if c != A and c != B])
        dac, dbc = D[A, C], D[B, C]
        duc = ((dac + dbc) - dab) * 0.5
        R[C] = ((R[C] - dac) - dbc) + duc
        D[A, C] = duc
        D[C, A] = duc
        R[A] = (((ra - dab) + (rb - dab)) - (k - 2) * dab) * 0.5
        node[A] = u
        active.pop(b)
    x, y, z = active
    root = 2 * n - 3
    for v, l in ((x, ((D[x, y] + D[x, z]) - D[y, z]) * 0.5), (y, ((D[x, y] + D[y, z]) - D[x, z]) * 0.5),
                 (z, ((D[x, z] + D[y, z]) - D[x, y]) * 0.5)):
        parent[node[v]], length[node[v]] = root, l
    return parent, length


def upper(D):
    """The upper triangle of a matrix, row-major."""
    return np.asarray(D, np.float64)[np.triu_indices(len(D), 1)]


def full(upper_values, n):
    D = np.zeros((n, n), np.float64)
    D[np.triu_indices(n, 1)] = upper_values
    return D + D.T


def core_matrix(codes, core_size):
    """d_ij = core_diff / core_size from the letter codes (0..3) of the rows."""
    N = codes.shape[0]
    same = np.zeros((N, N), np.int64)
    for x in range(4):
        m = (codes == x).astype(np.float64)
        same += np.rint(m @ m.T).astype(np.int64)
    diff = codes.shape[1] - same
    return diff.astype(np.float64) / float(core_size)


def acc_matrix(presence, core_genes):
    """d_ij = 1 - (inter + core_genes) / (uni + core_genes), 0 where the denominator is 0."""
    p = presence.astype(np.float64)
    inter = np.rint(p @ p.T)
    cnt = p.sum(axis=1)
    uni = cnt[:, None] + cnt[None, :] - inter
    den = uni + float(core_genes)
    with np.errstate(invalid="ignore", divide="ignore"):
        d = 1.0 - ((inter + float(core_genes)) / den)
    d[den == 0] = 0.0
    np.fill_diagonal(d, 0.0)
    return d


def leaf_sets(parent, n_leaves):
    below = [frozenset([k]) if k < n_leaves else frozenset() for k in range(len(parent))]
    for k in range(len(parent) - 1):
        below[int(parent[k])] = below[int(parent[k])] | below[k]
    return below


def splits(parent, n_leaves):
    """The distinct non-trivial bipartitions, each as the side without leaf 0."""
    everything = frozenset(range(n_leaves))
    out = set()
    for S in leaf_sets(parent, n_leaves)[:-1]:
        side = everything - S if 0 in S else S
        if 2 <= len(side) <= n_leaves - 2:
            out.add(side)
    return out


def compare_splits(a, b, n_leaves):
    A, B = splits(a, n_leaves), splits(b, n_leaves)
    return len(A), len(B), len(A & B)


def newick(parent, length, n_leaves):
    """pansim_tree_newick's text: leaves ind_<i>, children by smallest leaf, lengths %.17g."""
    n = len(parent)
    root = n - 1
    minleaf = [k if k < n_leaves else NONE for k in range(n)]
    kids = [[] for _ in range(n)]
    for k in range(root):
        minleaf[int(parent[k])] = min(minleaf[int(parent[k])], minleaf[k])
        kids[int(parent[k])].append(k)
    for v in kids:
        v.sort(key=lambda k: (minleaf[k], k))
    out = []
    stack = [(root, 0)]
    out.append(f"ind_{root}" if root < n_leaves else "(")
    while stack:
        v, i = stack[-1]
        if v >= n_leaves and i < len(kids[v]):
            if i:
                out.append(",")
            ch = kids[v][i]
            stack[-1] = (v, i + 1)
            out.append(f"ind_{ch}" if ch < n_leaves else "(")
            stack.append((ch, 0))
            continue
        if v >= n_leaves:
            out.append(")")
        if v != root:
            out.append(":%.17g" % length[v])
        stack.pop()
    return "".join(out) + ";\n"


def random_binary_tree(rng, n_leaves, caterpillar=False):
    """(parent, positive edge lengths) of a random rooted binary tree renumbered so that parents come after children."""
    live = list(range(n_leaves))
    parent = [NONE] * n_leaves
    nxt = n_leaves
    while len(live) > 1:
        if caterpillar:
            pick = [0, 1]
        else:
            pick = sorted(rng.choice(len(live), 2, replace=False).tolist())
        for i in reversed(pick):
            parent[live.pop(i)] = nxt
        parent.append(NONE)
        live.insert(0, nxt) if caterpillar else live.append(nxt)
        nxt += 1
    length = rng.uniform(0.05, 1.0, len(parent))
    length[-1] = 0.0
    return np.array(parent, np.uint32), length


def tree_metric(parent, length, n_leaves):
    """Path lengths between the leaves (the additive metric of the tree)."""
    n = len(parent)
    depth = np.zeros(n)
    for v in range(n - 2, -1, -1):
        depth[v] = depth[int(parent[v])] + length[v]
    paths = []
    for leaf in range(n_leaves):
        p, v = [leaf], leaf
        while int(parent[v]) != NONE:
            v = int(parent[v])
            p.append(v)
        paths.append(p)
    D = np.zeros((n_leaves, n_leaves))
    for i in range(n_leaves):
        si = set(paths[i])
        for j in range(i + 1, n_leaves):
            lca = next(v for v in paths[j] if v in si)
            D[i, j] = D[j, i] = depth[i] + depth[j] - 2 * depth[lca]
    return D
