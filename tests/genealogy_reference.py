"""numpy reference of the clonal genealogy (include/pansim_b200.h), written straight from the definitions: a loop over
the recorded generations that groups the live lineages by their parent, and the lowest common ancestor for the TMRCA."""
import numpy as np

NONE = 0xFFFFFFFF


def np_genealogy(H, N):
    """H: [T, N] parent vectors, oldest first. Returns (parent, individual, time, lineages_at_start) of the node table."""
    H = np.asarray(H, np.int64).reshape(-1, N)
    T = len(H)
    parent = [NONE] * N
    individual = list(range(N))
    time = [0] * N
    # live lineages at generation t: (smallest leaf below, node, ancestor a_t)
    lin = [(i, i, i) for i in range(N)]
    t = T
    while t >= 1 and len(lin) > 1:
        groups = {}
        for leaf, node, a in lin:
            groups.setdefault(int(H[t - 1][a]), []).append((leaf, node))
        nxt = []
        for x, members in sorted(groups.items(), key=lambda kv: min(m[0] for m in kv[1])):
            leaf = min(m[0] for m in members)
            if len(members) >= 2:                       # |{a_t(i) : a_{t-1}(i) = x}| >= 2: a node at generation t - 1
                nid = len(parent)
                parent.append(NONE)
                individual.append(x)
                time.append(T - (t - 1))
                for _, node in members:
                    parent[node] = nid
                nxt.append((leaf, nid, x))
            else:
                nxt.append((leaf, members[0][1], x))
        lin = nxt
        t -= 1
    if len(lin) > 1:                                    # not coalesced within the record: the virtual root
        nid = len(parent)
        parent.append(NONE)
        individual.append(NONE)
        time.append(T)
        for _, node, _ in lin:
            parent[node] = nid
    return (np.array(parent, np.uint32), np.array(individual, np.uint32), np.array(time, np.uint32),
            len(lin) if len(lin) > 1 else 1)


def np_tmrca_lca(parent, time, r1, r2):
    """Time of the lowest common ancestor of leaves r1[k] and r2[k] in the node table."""
    out = np.empty(len(r1), np.uint32)
    for k, (i, j) in enumerate(zip(r1, r2)):
        up = set()
        u = int(i)
        while u != NONE:
            up.add(u)
            u = int(parent[u])
        v = int(j)
        while v not in up:
            v = int(parent[v])
        out[k] = time[v]
    return out


def np_tmrca_walk(H, N, r1, r2):
    """Brute force, no tree: follow both lineages back through the record until they meet; T if they never do."""
    H = np.asarray(H, np.int64).reshape(-1, N)
    T = len(H)
    a = np.asarray(r1, np.int64).copy()
    b = np.asarray(r2, np.int64).copy()
    out = np.where(a == b, 0, T).astype(np.int64)
    open_ = a != b
    for t in range(T, 0, -1):
        a = H[t - 1][a]
        b = H[t - 1][b]
        met = open_ & (a == b)
        out[met] = T - (t - 1)
        open_ &= ~met
    return out.astype(np.uint32)


def parse_newick(text):
    """Newick text of the formatter -> (parent, branch length, leaves). Nodes are ("l", i) for leaf ind_<i> and
    ("i", k) for the k-th internal node opened; the root has no parent entry."""
    assert text.endswith(";\n")
    s = text[:-2]
    parent, length, leaves = {}, {}, []
    stack, last, n_internal, pos = [], None, 0, 0
    while pos < len(s):
        c = s[pos]
        if c == "(":
            node = ("i", n_internal)
            n_internal += 1
            if stack:
                parent[node] = stack[-1]
            stack.append(node)
            pos += 1
        elif c == ")":
            last = stack.pop()
            pos += 1
        elif c == ",":
            pos += 1
        elif c == ":":
            end = pos + 1
            while end < len(s) and s[end].isdigit():
                end += 1
            length[last] = int(s[pos + 1:end])
            pos = end
        else:
            end = pos
            while end < len(s) and s[end] not in ",():":
                end += 1
            assert s[pos:end].startswith("ind_"), s[pos:end]
            last = ("l", int(s[pos + 4:end]))
            leaves.append(last[1])
            if stack:
                parent[last] = stack[-1]
            pos = end
    assert not stack
    return parent, length, leaves


def newick_tmrca(text, r1, r2):
    """TMRCA of leaf pairs read from a Newick text: the height of their lowest common ancestor above the leaves."""
    parent, length, _ = parse_newick(text)
    height = {node: 0 for node in parent if node[0] == "l"}
    changed = True
    while changed:
        changed = False
        for node, p in parent.items():
            if node in height and p not in height:
                height[p] = height[node] + length[node]
                changed = True
    out = []
    for i, j in zip(r1, r2):
        a, b = ("l", int(i)), ("l", int(j))
        up = {a}
        while a in parent:
            a = parent[a]
            up.add(a)
        while b not in up:
            b = parent[b]
        out.append(height.get(b, 0))
    return np.array(out, np.uint32)
