"""Synthetic level-1 networks and their clique-tree plans (BASELINE.json configs 4-5).

Host-side harness code: integer / graph work only, no belief arithmetic.  In
production the arrays below come from the Julia side (cluster graph,
scopeindex maps, spanning-tree schedule, node families: INTEGRATION.md).  The
reference's own graph layer is O(n^2) in network size (allocatebeliefs:
src/beliefs.jl:521,526,536; triangulate_minfill!: src/clustergraph.jl:91-93),
so for 10^4-10^5 tips the clique tree is built directly, in linear time:

  network   Yule tree (rate 1, edge lengths floored at `min_len`) with `ntips`
            tips; `nretic` reticulations, each on a distinct internal node u
            with child edges (u,a), (u,b): both are subdivided by new nodes x, y
            and a hybrid edge x -> y is added (gamma ~ U(0.1,0.5), length
            U(0.01,0.1); the major edge u -> y gets 1-gamma).  Cycles {u,x,y} are
            vertex-disjoint triangles => level-1, moral graph already chordal.
  cliques   one cluster per node family {v} + parents(v), except the family
            {x,u}, which is inside {y,x,u}.  Nodes inside a cluster are listed by
            decreasing preorder index (src/clustergraph.jl:764-769).
  tree      cluster C_v hangs below the cluster that introduces its top-most
            parent; clusters holding the root hang below the first of them.

`plan_dict()` returns the same dictionary layout as workloads/*.json (what
ClusterGraphPlan / the C oracle take), plus the network tables needed to
simulate traits and to rebuild the network inside the oracle for cross-checks.
"""
from __future__ import annotations

import numpy as np


def level1_network(ntips, nretic, seed, min_len=0.01):
    """Returns dict(parents=[[(parent, length, gamma, edge_number)]], leaf=[bool], nnodes) with nodes
    numbered in a preorder (root = 0; every parent before its children; a hybrid after both parents).
    A hybrid's parents are listed minor (x) first, then major (u)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    if ntips < 2:
        raise ValueError("need at least 2 tips")
    # ---- Yule tree: node ids in creation order, root = 0; split[v] = time at which v splits
    par, kids, split, active, t = [-1], [[]], [None], [0], 0.0
    while len(active) < ntips:
        k = len(active)
        t += rng.exponential(1.0 / k)
        i = int(rng.integers(k))
        v = active[i]
        c1, c2 = len(par), len(par) + 1
        par += [v, v]
        kids += [[], []]
        split += [None, None]
        kids[v] = [c1, c2]
        split[v] = t
        active[i] = c1
        active.append(c2)
    t_end = t + rng.exponential(1.0 / len(active))
    n0 = len(par)
    split = [t_end if s_ is None else s_ for s_ in split]
    length = [0.0] + [max(split[v] - split[par[v]], min_len) for v in range(1, n0)]
    # general DAG tables: parents[v] = [(parent, length, gamma)]
    parents = [[] if v == 0 else [(par[v], length[v], 1.0)] for v in range(n0)]
    children = [list(k) for k in kids]
    internal = [v for v in range(n0) if kids[v]]
    if nretic > len(internal):
        raise ValueError("more reticulations than internal nodes")
    chosen = rng.choice(len(internal), size=nretic, replace=False) if nretic else []
    for ci in sorted(int(c) for c in chosen):
        u = internal[ci]
        a, b = kids[u]
        if rng.random() < 0.5:
            a, b = b, a
        x, y = len(parents), len(parents) + 1
        la, lb = parents[a][0][1], parents[b][0][1]
        fa, fb = rng.uniform(0.25, 0.75), rng.uniform(0.25, 0.75)
        gam = rng.uniform(0.1, 0.5)
        lh = rng.uniform(0.01, 0.1)
        parents.append([(u, max(la * fa, min_len), 1.0)])                      # x
        parents.append([(x, lh, gam), (u, max(lb * fb, min_len), 1.0 - gam)])  # y (hybrid): minor, major
        parents[a] = [(x, max(la * (1 - fa), min_len), 1.0)]
        parents[b] = [(y, max(lb * (1 - fb), min_len), 1.0)]
        children.append([a, y])   # x
        children.append([b])      # y
        children[u] = [x, y]
    n = len(parents)
    # ---- preorder: LIFO stack, a hybrid is pushed once all its parents are visited
    order, seen, stack = [], [0] * n, [0]
    while stack:
        v = stack.pop()
        order.append(v)
        for c in children[v]:
            seen[c] += 1
            if seen[c] == len(parents[c]):
                stack.append(c)
    assert len(order) == n
    new = [0] * n
    for i, v in enumerate(order):
        new[v] = i
    out_par, leaf, eno = [None] * n, [False] * n, 0
    for v in order:
        pl = []
        for (q, L, g) in parents[v]:
            eno += 1
            pl.append((new[q], float(L), float(g), eno))
        out_par[new[v]] = pl
        leaf[new[v]] = not children[v]
    return dict(parents=out_par, leaf=leaf, nnodes=n)


def edge_colors(net, ncolors):
    """Rate colour of every edge (by edge number): clades below the first `ncolors` nodes found
    breadth-first from the root get colours 0..ncolors-1; edges above them get colour 0."""
    n = net["nnodes"]
    children = [[] for _ in range(n)]
    for v in range(n):
        for (q, _, _, _) in net["parents"][v]:
            children[q].append(v)
    frontier = [0]
    while len(frontier) < ncolors:
        # split the first frontier node that has children
        k = next((i for i, v in enumerate(frontier) if children[v]), None)
        if k is None:
            break
        v = frontier.pop(k)
        frontier.extend(c for c in children[v] if c not in frontier)
    color_of_node = [0] * n
    for col, r in enumerate(frontier[:ncolors]):
        stack = [r]
        while stack:
            v = stack.pop()
            if color_of_node[v] == 0 or v == r:
                color_of_node[v] = col
                stack.extend(children[v])
    col = {}
    for v in range(n):
        for (q, _, _, e) in net["parents"][v]:
            col[e] = color_of_node[v]
    return col


def cliquetree_plan(net, ntraits, root_fixed=True, edge_color=None, name="synthetic"):
    """Direct clique tree of a network made by level1_network + everything a plan needs."""
    n, p = net["nnodes"], int(ntraits)
    parents, leaf = net["parents"], net["leaf"]
    fixed = [leaf[v] or (v == 0 and root_fixed) for v in range(n)]
    # x nodes: tree node v whose parent u also is a parent of a hybrid child of v
    sub = [-1] * n
    for y in range(n):
        if len(parents[y]) == 2:
            q = sorted(pp[0] for pp in parents[y])
            lo, hi = q  # lo = u (smaller preorder index), hi = x
            if len(parents[hi]) == 1 and parents[hi][0][0] == lo:
                sub[hi] = y
        elif len(parents[y]) > 2:
            raise ValueError("only hybrids with two parents are generated")
    clusters, cl_of = [], [-1] * n
    for v in range(1, n):
        if sub[v] >= 0:
            continue
        cl_of[v] = len(clusters)
        clusters.append(sorted([v] + [pp[0] for pp in parents[v]], reverse=True))
    for v in range(1, n):
        if sub[v] >= 0:
            cl_of[v] = cl_of[sub[v]]
    hub = next(c for c, nodes in enumerate(clusters) if 0 in nodes)
    cl_of[0] = hub
    nc = len(clusters)
    # tree edges: cluster c (introducing v) -> owner of its top-most (smallest-index) parent
    up = [-1] * nc
    sepnodes = [None] * nc
    for v in range(1, n):
        if sub[v] >= 0:
            continue
        c = cl_of[v]
        if c == hub:
            continue
        top = min(pp[0] for pp in parents[v])
        up[c] = cl_of[top]
        sepnodes[c] = [top]
    # edges in (min,max) lexicographic order = edge_labels order of the reference's MetaGraph
    edges = sorted((min(c, up[c]), max(c, up[c]), c) for c in range(nc) if up[c] >= 0)
    sepset_clusters = [[a, b] for a, b, _ in edges]
    sepset_nodes = [sepnodes[c] for _, _, c in edges]

    def scope_offsets(nodes):
        off, o = {}, 0
        for q in nodes:
            if not fixed[q]:
                off[q] = o
                o += p
        return off, o

    cl_off, belief_dim = [], []
    for nodes in clusters:
        off, m = scope_offsets(nodes)
        cl_off.append(off)
        belief_dim.append(m)
    upind = []
    for (a, b, _), sn in zip(edges, sepset_nodes):
        ua = [cl_off[a][q] + t for q in sn if not fixed[q] for t in range(p)]
        ub = [cl_off[b][q] + t for q in sn if not fixed[q] for t in range(p)]
        upind.append([ua, ub])
        belief_dim.append(len(ua))
    # schedule: DFS preorder of the clique tree from the hub (children by increasing cluster index)
    kids = [[] for _ in range(nc)]
    for c in range(nc):
        if up[c] >= 0:
            kids[up[c]].append(c)
    tp, tc, stack = [], [], [hub]
    while stack:
        c = stack.pop()
        if up[c] >= 0:
            tp.append(up[c])
            tc.append(c)
        stack.extend(reversed(kids[c]))
    assert len(tp) == nc - 1
    # node families (same table as pgbp_b200.families_table)
    tips = [v for v in range(n) if leaf[v]]
    row = {v: i for i, v in enumerate(tips)}
    mem_off, mem_pos, mem_len, mem_gam, mem_col, mem_par, datarow = [0], [], [], [], [], [], []
    for v in range(n):
        fam = [(v, 0.0, 1.0, 0)] + sorted(parents[v], key=lambda t: -t[0])
        off = cl_off[cl_of[v]]
        for k, (q, L, g, e) in enumerate(fam):
            mem_par.append(q if k else -1)
            mem_pos.append(-1 if fixed[q] else off[q])
            mem_len.append(L if k else 0.0)
            mem_gam.append(g if k else 1.0)
            mem_col.append((edge_color[e] if edge_color else 0) if k else 0)
        mem_off.append(len(mem_pos))
        datarow.append(row.get(v, -1))
    families = dict(nnodes=n, ntips=len(tips), root_fixed=int(bool(root_fixed)), node_cluster=list(cl_of),
                    mem_off=mem_off, mem_pos=mem_pos, mem_length=mem_len, mem_gamma=mem_gam, mem_color=mem_col,
                    node_datarow=datarow, mem_parent=mem_par)
    return dict(name=name, ntraits=p, nclusters=nc, belief_dim=belief_dim, sepset_clusters=sepset_clusters,
                upind=upind, trees=[[tp, tc]], families=families, root_cluster=hub,
                simulate=[[[q, L, g] for (q, L, g, _) in parents[v]] for v in range(n)], tip_nodes=tips,
                cluster_nodes=clusters, sepset_nodes=sepset_nodes, nnodes=n)


def simulate_tips(plan, R_of_edge, B, seed, mu=None):
    """Traits simulated down the network: X_v = sum_k gamma_k X_pa_k + N(0, sum_k gamma_k^2 t_k R_k).
    R_of_edge(v, k) -> p x p rate of the k-th parent edge of node v.  Returns [B][ntips][p]."""
    rng = np.random.Generator(np.random.PCG64(seed))
    p = plan["ntraits"]
    sim = plan["simulate"]
    n = len(sim)
    X = np.zeros((n, B, p))
    if mu is not None:
        X[0] = np.asarray(mu, dtype=float)
    cache = {}
    for v in range(1, n):
        var = np.zeros((p, p))
        mean = np.zeros((B, p))
        for k, (q, t, g) in enumerate(sim[v]):
            var += g * g * t * R_of_edge(v, k)
            mean += g * X[q]
        key = var.tobytes()
        L = cache.get(key)
        if L is None:
            L = np.linalg.cholesky(var)
            if len(cache) < 4096:
                cache[key] = L
        X[v] = mean + rng.normal(size=(B, p)) @ L.T
    return np.ascontiguousarray(X[plan["tip_nodes"]].transpose(1, 0, 2))
