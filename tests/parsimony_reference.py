"""numpy restatement of the parsimony definitions of include/pansim_b200.h: Hartigan's (1973) sets and scores on a
node table, vectorised over the characters, the fixed-rule reconstruction, the per-branch changes and the summary.

The tree is parent[n_nodes]: leaves 0 .. N-1, every parent id above its child's, the root last with parent
0xFFFFFFFF, every internal node with at least two children. A node's set is a bit mask of states per character."""
import numpy as np

NONE = 0xFFFFFFFF


def validate(parent, n_leaves: int):
    """Raise ValueError where the table breaks a rule of the definition."""
    parent = np.asarray(parent, np.int64)
    n, N = len(parent), n_leaves
    if n < N or n > 2 * N - 1:
        raise ValueError(f"{n} nodes for {N} leaves")
    if parent[-1] != NONE:
        raise ValueError("the last node is not the root")
    k = np.arange(n - 1)
    p = parent[:-1]
    if ((p <= k) | (p < N) | (p >= n)).any():
        raise ValueError("a parent is not an internal node with a larger id")
    kids = np.bincount(p, minlength=n)[N:]
    if (kids < 2).any():
        raise ValueError("an internal node has fewer than two children")


def children(parent, n_leaves: int):
    """The children of each internal node N + v, ascending."""
    parent = np.asarray(parent, np.int64)
    out = [[] for _ in range(len(parent) - n_leaves)]
    for k, p in enumerate(parent[:-1].tolist()):
        out[p - n_leaves].append(k)
    return out


def hartigan(parent, leaf_states, n_states: int):
    """leaf_states: int [N, C]. Returns (score int64 [C], state int8 [n_nodes, C] of the reconstruction,
    changed bool [n_nodes, C]: the state at the node differs from its parent's; False at the root)."""
    validate(parent, leaf_states.shape[0])
    parent = np.asarray(parent, np.int64)
    N, C = leaf_states.shape
    n = len(parent)
    sets = np.zeros((n, C), np.uint8)
    sets[:N] = (1 << leaf_states.astype(np.uint8)).astype(np.uint8)
    score = np.zeros(C, np.int64)
    kids = children(parent, N)
    for v, ch in enumerate(kids):
        cnt = np.stack([sum(((sets[u] >> x) & 1).astype(np.int64) for u in ch) for x in range(n_states)])
        m = cnt.max(axis=0)
        sets[N + v] = sum(((cnt[x] == m).astype(np.uint8) << x) for x in range(n_states))
        score += len(ch) - m

    def lowest(s):
        out = np.zeros(s.shape, np.int8)
        for x in range(n_states - 1, -1, -1):
            out = np.where((s >> x) & 1, np.int8(x), out)
        return out

    state = np.zeros((n, C), np.int8)
    state[:N] = leaf_states
    changed = np.zeros((n, C), bool)
    state[n - 1] = lowest(sets[n - 1]) if n > N else state[n - 1]
    for v in range(n - 2, N - 1, -1):
        ps = state[parent[v]]
        inset = ((sets[v] >> ps.astype(np.uint8)) & 1).astype(bool)
        state[v] = np.where(inset, ps, lowest(sets[v]))
    for v in range(n - 1):
        changed[v] = state[v] != state[parent[v]]
    return score, state, changed


def summary(score, leaf_states, n_states: int):
    """(characters, variable, tree_length, min_changes, max_changes, homoplastic) of the definition."""
    N, C = leaf_states.shape
    counts = np.stack([(leaf_states == x).sum(axis=0) for x in range(n_states)])
    distinct = (counts > 0).sum(axis=0)
    return (C, int((distinct >= 2).sum()), int(score.sum()), int((distinct - 1).sum()), int((N - counts.max(axis=0)).sum()),
            int((score > distinct - 1).sum()))


def indices(s):
    """(CI, RI) of a summary tuple, NaN for a zero denominator."""
    _, _, S, M, G, _ = s
    ci = M / S if S else float("nan")
    ri = (G - S) / (G - M) if G != M else float("nan")
    return ci, ri


def core_parsimony(parent, core_codes):
    """core_codes: uint8 [N, L] letter codes 0..3 (A, C, G, T). Returns (summary, site scores, branch changes)."""
    score, _, changed = hartigan(parent, core_codes, 4)
    return summary(score, core_codes, 4), score.astype(np.uint32), changed.sum(axis=1).astype(np.uint64)


def gene_parsimony(parent, presence):
    """presence: bool/uint8 [N, G]. Returns (summary, gene scores, gains, losses)."""
    pres = np.asarray(presence).astype(np.int8)
    score, state, changed = hartigan(parent, pres, 2)
    parent = np.asarray(parent, np.int64)
    gains = np.zeros(len(parent), np.uint64)
    losses = np.zeros(len(parent), np.uint64)
    gains[:-1] = (changed[:-1] & (state[:-1] == 1)).sum(axis=1)
    losses[:-1] = (changed[:-1] & (state[:-1] == 0)).sum(axis=1)
    return summary(score, pres, 2), score.astype(np.uint32), gains, losses


def random_tree(rng, n_leaves: int, max_children: int = 4):
    """A random rooted tree over the leaves, renumbered in postorder: merges random groups of 2..max_children of the
    live lineages until one is left."""
    live = list(range(n_leaves))
    parent = [NONE] * n_leaves
    nxt = n_leaves
    while len(live) > 1:
        k = int(rng.integers(2, min(max_children, len(live)) + 1))
        pick = rng.choice(len(live), k, replace=False)
        for i in sorted(pick.tolist(), reverse=True):
            parent[live.pop(i)] = nxt
        parent.append(NONE)
        live.append(nxt)
        nxt += 1
    return np.array(parent, np.uint32)
