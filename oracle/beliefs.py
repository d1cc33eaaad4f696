"""Belief state and factor initialisation.  Restates src/beliefs.jl (canonical
form only; GeneralizedBelief is out of scope).

TEST INFRASTRUCTURE (see oracle/__init__.py).

Trait data: `tbl` is an (ntaxa x ntraits) float array, NaN = missing, rows in
the order of `taxa` (the reference takes a Tables.ColumnTable).
All node / cluster indices exposed here are 1-based like the reference's.
"""
from __future__ import annotations

import numpy as np

from .canonical import marginalize

CLUSTER, SEPSET = 1, 2


class CanonicalBelief:
    """src/beliefs.jl:72-132.  inscope: bool (ntraits x nnodes)."""

    def __init__(self, nodelabel, ntraits, inscope, btype, metadata):
        self.nodelabel = list(nodelabel)
        self.ntraits = int(ntraits)
        self.inscope = np.asarray(inscope, dtype=bool).reshape(ntraits, len(self.nodelabel))
        m = int(self.inscope.sum())
        self.mu = np.zeros(m)
        self.h = np.zeros(m)
        self.J = np.zeros((m, m))
        self.g = 0.0
        self.type = btype
        self.metadata = metadata

    def dimension(self):
        return int(self.inscope.sum())

    def nodedimensions(self):
        return self.inscope.sum(axis=0).astype(int)

    def copy(self):
        b = CanonicalBelief(self.nodelabel, self.ntraits, self.inscope.copy(), self.type, self.metadata)
        b.mu, b.h, b.J, b.g = self.mu.copy(), self.h.copy(), self.J.copy(), self.g
        return b


class ClusterFactor:
    """src/beliefs.jl:6-16, 604-609."""

    def __init__(self, belief: CanonicalBelief):
        self.h, self.J, self.g = belief.h.copy(), belief.J.copy(), belief.g
        self.metadata = belief.metadata


class MessageResidual:
    """src/beliefs.jl:895-924."""

    def __init__(self, J, h):
        self.dh = np.zeros_like(h)
        self.dJ = np.zeros_like(J)
        empty = h.size == 0
        self.kldiv = 0.0 if empty else -1.0
        self.iscalibrated_resid = bool(empty)
        self.iscalibrated_kl = bool(empty)

    def reset_flags(self, resetkl: bool):
        """src/beliefs.jl:973-979."""
        if self.dh.size == 0:
            return
        if resetkl:
            self.kldiv = -1.0
        self.iscalibrated_resid = False
        self.iscalibrated_kl = False


# --------------------------------------------------------------------------
# scopeindex (src/beliefs.jl:334-436) -- all return 0-based numpy int arrays
# --------------------------------------------------------------------------
def scopeindex_nodes(node_labels, belief: CanonicalBelief):
    """src/beliefs.jl:354-373."""
    nd = belief.nodedimensions()
    cs = np.concatenate([[0], np.cumsum(nd)])
    res = []
    for lab in node_labels:
        if lab not in belief.nodelabel:
            raise ValueError("some label is not in the belief's node labels")
        jj = belief.nodelabel.index(lab)
        res.extend(range(cs[jj], cs[jj] + nd[jj]))
    return np.array(res, dtype=np.int64)


def scopeindex(sep: CanonicalBelief, clu: CanonicalBelief):
    """src/beliefs.jl:389-405."""
    ni = []
    for lab in sep.nodelabel:
        if lab not in clu.nodelabel:
            raise ValueError("subset_labels not a subset of belief_labels")
        ni.append(clu.nodelabel.index(lab))
    if any(ni[k] > ni[k + 1] for k in range(len(ni) - 1)):
        raise ValueError("subset labels come in a different order in the belief")
    if np.any(sep.inscope & ~clu.inscope[:, ni]):
        raise ValueError("some variable(s) in subset's scope yet not in full belief's scope")
    sub = np.zeros_like(clu.inscope)
    sub[:, ni] = sep.inscope
    # column-major vectorisation restricted to the cluster's in-scope entries
    return np.flatnonzero(sub.T[clu.inscope.T]).astype(np.int64)


def scopeindex_node(node_lab, sep: CanonicalBelief, clu: CanonicalBelief):
    """src/beliefs.jl:418-436 -> (ind_in_sepset, ind_in_cluster) of the shared
    in-scope traits of one node."""
    s_j = sep.nodelabel.index(node_lab)
    c_j = clu.nodelabel.index(node_lab)
    s_node = sep.inscope[:, s_j]
    if np.any(s_node & ~clu.inscope[:, c_j]):
        raise ValueError("some traits are in sepset's but not in cluster's scope")
    s_insc = np.zeros_like(sep.inscope)
    s_insc[:, s_j] = s_node
    c_insc = np.zeros_like(clu.inscope)
    c_insc[:, c_j] = s_node
    return (np.flatnonzero(s_insc.T[sep.inscope.T]).astype(np.int64),
            np.flatnonzero(c_insc.T[clu.inscope.T]).astype(np.int64))


# --------------------------------------------------------------------------
# allocatebeliefs (src/beliefs.jl:478-594)
# --------------------------------------------------------------------------
def allocatebeliefs(tbl, taxa, prenodes, cgraph, model):
    """Returns (beliefs, (node2cluster, node2family, node2fixed, node2degen,
    cluster2nodes)); indices 1-based; beliefs = clusters then sepsets."""
    tbl = np.asarray(tbl, dtype=float)
    numtraits = tbl.shape[1]
    nnodes = len(prenodes)
    fixedroot = model.isrootfixed()
    idx = {id(n): i + 1 for i, n in enumerate(prenodes)}
    taxa = list(taxa)
    clusterlabs = cgraph.labels
    node2cluster = [0] * nnodes
    node2family = [None] * nnodes
    node2fixed = [False] * nnodes
    node2degen = [False] * nnodes
    cluster2nodes = [[] for _ in clusterlabs]
    hasdata = np.zeros((numtraits, nnodes), dtype=bool)
    for ni in range(nnodes, 0, -1):
        node = prenodes[ni - 1]
        if node.leaf:
            if node.name not in taxa:
                raise ValueError(f"tip {node.name} in network without any data")
            hasdata[:, ni - 1] = ~np.isnan(tbl[taxa.index(node.name)])
        i_parents = []
        degen = True
        for e in node.edges:
            if e.child is node:
                if e.length > 0:
                    degen = False
                i_parents.append(idx[id(e.parent)])
            else:
                hasdata[:, ni - 1] |= hasdata[:, idx[id(e.child)] - 1]
        i_parents.sort(reverse=True)
        nf = [ni] + i_parents
        ci = next((c for c, lab in enumerate(clusterlabs, start=1)
                   if set(nf) <= set(cgraph.vdata[lab][1])), None)
        if ci is None:
            raise ValueError(f"no cluster containing the node family for {node.name}.")
        node2cluster[ni - 1] = ci
        node2family[ni - 1] = nf
        if node.leaf or (ni == 1 and fixedroot):
            node2fixed[ni - 1] = True
        node2degen[ni - 1] = degen and ni > 1
        cluster2nodes[ci - 1].append(ni)
    if any(node2degen):
        raise NotImplementedError("degenerate node families (GeneralizedBelief) are out of scope")

    def build_inscope(nodeindices):
        insc = np.zeros((numtraits, len(nodeindices)), dtype=bool)
        for i, ni in enumerate(nodeindices):
            node = prenodes[ni - 1]
            if node.leaf or (ni == 1 and fixedroot):
                continue
            insc[:, i] = hasdata[:, ni - 1]
        return insc

    beliefs = []
    for lab in clusterlabs:
        ninds = cgraph.vdata[lab][1]
        beliefs.append(CanonicalBelief(ninds, numtraits, build_inscope(ninds), CLUSTER, lab))
    for (l1, l2) in cgraph.edge_labels():
        ninds = cgraph.sepset(l1, l2)
        beliefs.append(CanonicalBelief(ninds, numtraits, build_inscope(ninds), SEPSET, (l1, l2)))
    return beliefs, (node2cluster, node2family, node2fixed, node2degen, cluster2nodes)


# --------------------------------------------------------------------------
# absorbevidence / absorbleaf (src/beliefupdates.jl:210-231, 266-274)
# --------------------------------------------------------------------------
def absorbevidence(h, J, g, dataindex, datavalues):
    """dataindex 0-based.  Returns ((h,J,g), missingdata_indices) where the
    latter index the reduced system."""
    dataindex = np.asarray(dataindex, dtype=np.int64)
    datavalues = np.asarray(datavalues, dtype=float)
    hasd = ~np.isnan(datavalues)
    absorb = dataindex[hasd]
    nvar = h.size
    keep = np.setdiff1d(np.arange(nvar), absorb)
    missing_idx = np.array([int(np.flatnonzero(keep == i)[0]) for i in dataindex[~hasd]], dtype=np.int64)
    data_nm = datavalues[hasd]
    if absorb.size == 0:
        return (h, J, g), missing_idx
    Jk_data = J[np.ix_(keep, absorb)] @ data_nm
    Ja_data = J[np.ix_(absorb, absorb)] @ data_nm
    g = g + float(h[absorb] @ data_nm) - float(Ja_data @ data_nm) / 2
    hk = h[keep] - Jk_data
    return (hk, J[np.ix_(keep, keep)], g), missing_idx


def absorbleaf(h, J, g, row):
    """src/beliefupdates.jl:266-274: the leaf's traits are the first variables."""
    p = row.size
    (h, J, g), miss = absorbevidence(h, J, g, np.arange(p), row)
    if miss.size:
        keep = np.setdiff1d(np.arange(h.size), miss)
        h, J, g = marginalize(h, J, g, keep, miss)
    return h, J, g


# --------------------------------------------------------------------------
# assignfactors! (src/beliefs.jl:786-861)
# --------------------------------------------------------------------------
def init_beliefs_reset(beliefs):
    """src/beliefs.jl:706-717."""
    for b in beliefs:
        b.h[:] = 0
        b.J[:] = 0
        b.g = 0.0


def assignfactors(beliefs, model, tbl, taxa, prenodes, node2cluster, node2family, node2fixed):
    tbl = np.asarray(tbl, dtype=float)
    taxa = list(taxa)
    init_beliefs_reset(beliefs)
    p = model.ntraits
    for ni, ci in enumerate(node2cluster, start=1):
        be = beliefs[ci - 1]
        nf = node2family[ni - 1]
        ch = prenodes[ni - 1]
        if len(nf) == 1:
            if ni != 1:
                raise ValueError("only the root node can belong to a family of size 1")
            if node2fixed[0]:
                continue
            phi = model.factor_root()
        else:
            if len(nf) == 2:
                phi = model.factor_treeedge(ch.parent_edges()[0])
            else:
                pae = []
                for pi in nf[1:]:
                    for e in prenodes[pi - 1].edges:
                        if e.child is ch:
                            pae.append(e)
                            break
                phi = model.factor_hybridnode(pae)
            if node2fixed[ni - 1]:  # leaf
                phi = absorbleaf(*phi, tbl[taxa.index(ch.name)])
            if any(node2fixed[q - 1] for q in nf[1:]):  # a parent is the fixed root
                n = phi[0].size
                phi, _ = absorbevidence(*phi, np.arange(n - p, n), model.rootpriormeanvector())
        i_inscope = [q for q in nf if not node2fixed[q - 1]]
        factorind = scopeindex_nodes(i_inscope, be)
        h, J, g = phi
        if factorind.size != p * len(i_inscope):
            cols = [be.nodelabel.index(q) for q in i_inscope]
            var_inscope = be.inscope[:, cols]
            keep_index = np.flatnonzero(var_inscope.T.ravel())  # 0-based, column-major
            # DELIBERATE DEVIATION from src/beliefs.jl:845-857: a parent's out-of-scope trait t is observed
            # below no child of it, so the child's trait t is gone already (marginalised above, or by
            # absorbleaf); under Brownian motion the child's other traits depend on the parents' trait t
            # not at all, and its rows of (h, J) are zero in exact arithmetic.  They are dropped, not
            # marginalised: the reference factorises their roundoff (~1e-14 on short edges), which adds
            # ~ -log(1e-14)/2 per trait to g, or fails on a negative pivot.
            if not node2fixed[ni - 1]:
                kc = keep_index[keep_index < p]
                integ_ch = np.setdiff1d(np.arange(p), kc)
                keep_ch = np.setdiff1d(np.arange(h.size), integ_ch)
                h, J, g = marginalize(h, J, g, keep_ch, integ_ch)
                if any(not node2fixed[q - 1] for q in nf[1:]):
                    nkc = kc.size
                    keep_pa = keep_index[keep_index >= p] - (p - nkc)
                    keep = np.concatenate([np.arange(nkc), keep_pa])
                    h, J = h[keep], J[np.ix_(keep, keep)]
            else:
                h, J = h[keep_index], J[np.ix_(keep_index, keep_index)]
        # mult! (src/beliefupdates.jl:483-488)
        be.h[factorind] += h
        be.J[np.ix_(factorind, factorind)] += J
        be.g += g
    return None
