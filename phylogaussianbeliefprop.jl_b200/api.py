"""Host-side mirror of the reference's interface for the message-passing path.

Same names, argument meaning and error behaviour as
PhyloGaussianBeliefProp.jl (`PGBP.` prefix there), with every belief carrying
a leading batch axis of B independent replicas:

    reference (one replicate)                      here (B replicates)
    ------------------------------------------     ---------------------------------------------
    allocatebeliefs / init_beliefs_allocate        ClusterGraphPlan.from_beliefs(...) + BatchedClusterGraphBelief
    assignfactors! / init_factors_frommodel!       b.assignfactors(...)            src/beliefs.jl:786
    ClusterGraphBelief(b, ...)                     BatchedClusterGraphBelief(plan, B)
    calibrate!(b, sched, niter; auto, ...)         calibrate(b, sched, niter, auto=...) -> (succ[B], iscal[B])
    propagate_1traversal_postorder!(b, spt...)     propagate_1traversal_postorder(b, tree)
    propagate_belief!(to, sepset, from, resid)     propagate_belief(b, to, sepset, frm)
    integratebelief!(b, j)                         integratebelief(b, j) -> (mu[B,m], norm[B])
    factored_energy(b)                             factored_energy(b) -> [B,3]
    regularizebeliefs_bycluster!(b, cg) ...        regularizebeliefs_bycluster(b) ...
    init_beliefs_reset_fromfactors!(b)             init_beliefs_reset_fromfactors(b)

Indices are 1-based wherever the reference's are (belief / cluster indices,
schedule tuples), so the parity tests read like the reference's tests.  The
graph layer (cluster-graph construction, spanning trees) is NOT part of this
package: like the Julia wrapper (INTEGRATION.md) it consumes that layer's
output.  Nothing here computes beliefs on the CPU.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np

from . import _lib as L

_i32p = C.POINTER(C.c_int32)
_f64p = C.POINTER(C.c_double)


def _ia(x):
    a = np.ascontiguousarray(np.asarray(x, dtype=np.int32).ravel())
    return a, a.ctypes.data_as(_i32p)


def _fa(x):
    a = np.ascontiguousarray(np.asarray(x, dtype=np.float64).ravel())
    return a, a.ctypes.data_as(_f64p)


def _fptr(a):
    return None if a is None else a.ctypes.data_as(_f64p)


def scopeindex(sub_labels, sub_inscope, labels, inscope):
    """scopeindex(sepset, cluster) -- src/beliefs.jl:391-405, 0-based result.
    Pure index work (the reference recomputes it for every message; here it is
    computed once per plan)."""
    labels = list(labels)
    sub_inscope = np.asarray(sub_inscope, dtype=bool)
    inscope = np.asarray(inscope, dtype=bool)
    ni = []
    for lab in sub_labels:
        if lab not in labels:
            raise ValueError("subset_labels not a subset of belief_labels")
        ni.append(labels.index(lab))
    if any(ni[k] > ni[k + 1] for k in range(len(ni) - 1)):
        raise ValueError("subset labels come in a different order in the belief")
    if np.any(sub_inscope & ~inscope[:, ni]):
        raise ValueError("some variable(s) in subset's scope yet not in full belief's scope")
    sub = np.zeros_like(inscope)
    sub[:, ni] = sub_inscope
    return np.flatnonzero(sub.T[inscope.T]).astype(np.int32)


class ClusterGraphPlan:
    """Static description of one cluster graph + its schedules (pgbp_plan).

    belief_dim       [nclusters+nsepsets]
    sepset_clusters  [(a, b)] 0-based cluster indices, sepsets in edge_labels order
    upind            [(upind_a, upind_b)] 0-based scope maps
    trees            [(parent_idx, child_idx)] 0-based, edges in preorder
    families         optional dict for assignfactors (see from_beliefs)
    """

    def __init__(self, nclusters, belief_dim, sepset_clusters, upind, trees, ntraits, families=None, lib=None):
        self.lib = lib or L.default_library()
        self.nclusters = int(nclusters)
        self.belief_dim = [int(x) for x in belief_dim]
        self.nsepsets = len(self.belief_dim) - self.nclusters
        self.sepset_clusters = [(int(a), int(b)) for a, b in sepset_clusters]
        self.trees = [(list(map(int, p)), list(map(int, c))) for p, c in trees]
        self.upind = [([int(x) for x in ua], [int(x) for x in ub]) for ua, ub in upind]
        self.ntraits = int(ntraits)
        self.families = families
        keep = []  # keep numpy buffers alive during the call
        d = L.PlanDesc()
        d.nclusters, d.nsepsets, d.ntraits = self.nclusters, self.nsepsets, self.ntraits
        a, d.belief_dim = _ia(self.belief_dim); keep.append(a)
        a, d.sepset_clusters = _ia([x for ab in self.sepset_clusters for x in ab] or [0]); keep.append(a)
        off, flat = [0], []
        for ua, ub in upind:
            flat.extend(int(x) for x in ua); off.append(len(flat))
            flat.extend(int(x) for x in ub); off.append(len(flat))
        a, d.upind_off = _ia(off); keep.append(a)
        a, d.upind = _ia(flat or [0]); keep.append(a)
        d.ntrees = len(self.trees)
        toff, tp, tc = [0], [], []
        for p, c in self.trees:
            tp.extend(p); tc.extend(c); toff.append(len(tp))
        a, d.tree_off = _ia(toff); keep.append(a)
        a, d.tree_parent = _ia(tp or [0]); keep.append(a)
        a, d.tree_child = _ia(tc or [0]); keep.append(a)
        if families is not None:
            ft = L.FamilyTable()
            ft.nnodes, ft.ntips, ft.root_fixed = int(families["nnodes"]), int(families["ntips"]), int(families["root_fixed"])
            a, ft.node_cluster = _ia(families["node_cluster"]); keep.append(a)
            a, ft.mem_off = _ia(families["mem_off"]); keep.append(a)
            a, ft.mem_pos = _ia(families["mem_pos"]); keep.append(a)
            a, ft.mem_length = _fa(families["mem_length"]); keep.append(a)
            a, ft.mem_gamma = _fa(families["mem_gamma"]); keep.append(a)
            a, ft.mem_color = _ia(families["mem_color"]); keep.append(a)
            a, ft.node_datarow = _ia(families["node_datarow"]); keep.append(a)
            if families.get("mem_tpos") is not None:  # trait-level scopes (missing data)
                a, ft.mem_tpos = _ia(families["mem_tpos"]); keep.append(a)
                a = np.ascontiguousarray(np.asarray(families["tip_missing"], dtype=np.uint8)); keep.append(a)
                ft.tip_missing = a.ctypes.data_as(C.POINTER(C.c_uint8))
            keep.append(ft)
            d.families = C.pointer(ft)
        h = C.c_void_p()
        self.lib.check(self.lib.pgbp_plan_create(C.byref(d), C.byref(h)))
        self.handle = h

    def __del__(self):
        h = getattr(self, "handle", None)
        if h:
            self.lib.pgbp_plan_destroy(h)
            self.handle = None

    # ------------------------------------------------------------------
    @classmethod
    def from_beliefs(cls, beliefs, nclusters, cluster_labels, schedule=(), families=None, lib=None):
        """Build a plan from the reference's own objects: `beliefs` is the
        vector returned by allocatebeliefs (clusters first, then sepsets; each
        with .nodelabel, .inscope (ntraits x nnodes), .metadata), `schedule` a
        list of spanning trees as returned by spanningtree(s)_clusterlist
        (4-tuples, 1-based cluster indices)."""
        lab2idx = {lab: i for i, lab in enumerate(cluster_labels)}
        dims = [int(np.asarray(b.inscope).sum()) for b in beliefs]
        sc, up = [], []
        for s in beliefs[nclusters:]:
            l1, l2 = s.metadata
            a, b_ = lab2idx[l1], lab2idx[l2]
            sc.append((a, b_))
            up.append((scopeindex(s.nodelabel, s.inscope, beliefs[a].nodelabel, beliefs[a].inscope),
                       scopeindex(s.nodelabel, s.inscope, beliefs[b_].nodelabel, beliefs[b_].inscope)))
        trees = [([j - 1 for j in spt[2]], [j - 1 for j in spt[3]]) for spt in schedule]
        plan = cls(nclusters, dims, sc, up, trees, beliefs[0].ntraits, families, lib)
        plan.schedule = list(schedule)
        return plan

    def tree_id(self, spt):
        """Index of a spanning tree (reference 4-tuple or 0-based int)."""
        if isinstance(spt, (int, np.integer)):
            return int(spt)
        key = ([j - 1 for j in spt[2]], [j - 1 for j in spt[3]])
        for t, tr in enumerate(self.trees):
            if tr == key:
                return t
        raise ValueError("this spanning tree is not part of the plan's schedule")

    def levels(self, tree, direction):
        n, ns = C.c_int32(), C.c_int32()
        self.lib.check(self.lib.pgbp_plan_get_levels(self.handle, tree, direction, C.byref(n), C.byref(ns),
                                                     None, None, None, None, None))
        arr = [np.zeros(n.value, dtype=np.int32) for _ in range(5)]
        self.lib.check(self.lib.pgbp_plan_get_levels(self.handle, tree, direction, C.byref(n), C.byref(ns),
                                                     *[a.ctypes.data_as(_i32p) for a in arr]))
        return dict(nsteps=ns.value, ref=arr[0], step=arr[1], frm=arr[2], sepset=arr[3], to=arr[4])

    def traversal_cost(self, tree, direction, track_residuals=True):
        by, fl = C.c_double(), C.c_double()
        self.lib.check(self.lib.pgbp_plan_traversal_cost(self.handle, tree, direction, int(track_residuals),
                                                         C.byref(by), C.byref(fl)))
        return by.value, fl.value

    def belief_slot(self, belief):
        j, h, g = C.c_int64(), C.c_int64(), C.c_int64()
        self.lib.check(self.lib.pgbp_belief_slot(self.handle, belief, C.byref(j), C.byref(h), C.byref(g)))
        return j.value, h.value, g.value


def families_table(prenodes_info, node2cluster, node2family, node2fixed, beliefs, ntraits, root_fixed,
                   taxa=None, edge_color=None, tip_missing=None):
    """Node-family table for pgbp_assign_factors from the reference's
    allocatebeliefs outputs (node2cluster, node2family, node2fixed; 1-based) and
    per-node parent-edge data: prenodes_info[v] = dict(name, leaf,
    parents=[(parent_preorder_idx_1based, length, gamma, edge_number)]).
    tip_missing: optional (ntips, ntraits) boolean array, True where the trait is missing at that tip
    (row order = taxa); with it, or when some belief has a partial trait scope, the table carries the
    trait-level scope positions (mem_tpos) and the plan uses the scoped factor-assignment path."""
    n = len(node2cluster)
    taxa = list(taxa) if taxa is not None else None
    mem_off, mem_pos, mem_len, mem_gam, mem_col, datarow = [0], [], [], [], [], []
    mem_tpos, mem_par, partial = [], [], False
    for v in range(n):
        ci = node2cluster[v] - 1
        be = beliefs[ci]
        nf = node2family[v]
        info = prenodes_info[v]
        nd = np.asarray(be.inscope).sum(axis=0).astype(int)
        cs = np.concatenate([[0], np.cumsum(nd)])
        for k, q in enumerate(nf):
            if node2fixed[q - 1]:
                mem_pos.append(-1)
                mem_tpos.extend([-1] * ntraits)
            else:
                jj = list(be.nodelabel).index(q)
                if nd[jj] != ntraits:
                    partial = True
                mem_pos.append(int(cs[jj]))
                col = np.asarray(be.inscope)[:, jj].astype(bool)
                run = int(cs[jj])
                for t in range(ntraits):
                    if col[t]:
                        mem_tpos.append(run)
                        run += 1
                    else:
                        mem_tpos.append(-1)
            if k == 0:
                mem_len.append(0.0); mem_gam.append(1.0); mem_col.append(0); mem_par.append(-1)
            else:
                par = next(p for p in info["parents"] if p[0] == q)
                mem_len.append(float(par[1])); mem_gam.append(float(par[2])); mem_par.append(int(par[0]) - 1)
                mem_col.append(int(edge_color(par[3])) if edge_color else 0)
        mem_off.append(len(mem_pos))
        datarow.append(taxa.index(info["name"]) if (info["leaf"] and taxa is not None) else -1)
    out = dict(nnodes=n, ntips=len(taxa) if taxa is not None else 0, root_fixed=int(bool(root_fixed)),
               node_cluster=[c - 1 for c in node2cluster], mem_off=mem_off, mem_pos=mem_pos,
               mem_length=mem_len, mem_gamma=mem_gam, mem_color=mem_col, node_datarow=datarow, mem_parent=mem_par)
    tm = None if tip_missing is None else np.ascontiguousarray(np.asarray(tip_missing, dtype=bool).reshape(out["ntips"], ntraits))
    if partial or (tm is not None and tm.any()):
        out["mem_tpos"] = mem_tpos
        out["tip_missing"] = (tm if tm is not None else np.zeros((out["ntips"], ntraits), bool)).astype(np.uint8).ravel()
    return out


def bm_params(rates, mu, v=None):
    """Pack Brownian-motion parameters for assignfactors: rates = [R_c] (p x p
    each; a scalar / vector means univariate / diagonal), mu, v (None = fixed
    root).  Returns a flat float64 vector (one parameter set)."""
    mu = np.atleast_1d(np.asarray(mu, dtype=float))
    p = mu.size
    out = []
    for R in rates:
        R = np.asarray(R, dtype=float)
        if R.ndim == 0:
            R = R.reshape(1, 1)
        elif R.ndim == 1:
            R = np.diag(R)
        if R.shape != (p, p):
            raise ValueError("R and mu have conflicting sizes")
        out.append(R.T.ravel())  # column-major
    out.append(mu)
    if v is None:
        V = np.zeros((p, p))
    else:
        V = np.asarray(v, dtype=float)
        if V.ndim == 0:
            V = V.reshape(1, 1)
        elif V.ndim == 1:
            V = np.diag(V)
    out.append(V.T.ravel())
    return np.concatenate(out)


class BatchedClusterGraphBelief:
    """B replicas of a ClusterGraphBelief (src/clustergraphbeliefs.jl:26-53) on
    one GPU: beliefs, factors, message residuals and per-element status."""

    def __init__(self, plan: ClusterGraphPlan, B: int, device: int = 0, factors=True, residuals=True, stream=None,
                 shared_precision_group: int = 0):
        """shared_precision_group = g > 1: the g consecutive elements of a group are trait replicates under
        ONE parameter vector; their (identical) precisions J are stored and updated once per group."""
        self.plan, self.lib, self.B = plan, plan.lib, int(B)
        flags = (L.BATCH_FACTORS if factors else 0) | (L.BATCH_RESIDUALS if residuals else 0)
        h = C.c_void_p()
        self.lib.check(self.lib.pgbp_batch_create_shared(plan.handle, self.B, int(shared_precision_group), int(device),
                                                         flags, C.byref(h)))
        self.handle = h
        if stream is not None:
            self.lib.check(self.lib.pgbp_batch_set_stream(h, C.c_void_p(int(stream))))
        self.nclusters, self.nsepsets = plan.nclusters, plan.nsepsets

    def __del__(self):
        h = getattr(self, "handle", None)
        if h:
            self.lib.pgbp_batch_destroy(h)
            self.handle = None

    # -- sizes -----------------------------------------------------------
    def nbeliefs(self):
        return self.nclusters + self.nsepsets

    def dimension(self, j):
        return self.plan.belief_dim[j - 1]

    def device_bytes(self):
        return self.lib.pgbp_batch_device_bytes(self.handle)

    def belief_rows(self, j):
        """Rows (h first row, g row) of belief j (1-based) in the array device_view() returns: the plan's slots, or
        the compact numbering of a shared-precision batch."""
        h, g = C.c_int64(), C.c_int64()
        self.lib.check(self.lib.pgbp_batch_belief_rows(self.handle, j - 1, C.byref(h), C.byref(g)))
        return h.value, g.value

    def launch_count(self, reset=False):
        return self.lib.pgbp_batch_launch_count(self.handle, int(reset))

    def set_walk_mode(self, mode):
        """-1 auto, 0 level-parallel launches, 1 single walk kernel per traversal."""
        self.lib.check(self.lib.pgbp_batch_set_walk_mode(self.handle, int(mode)))

    def set_pipeline(self, nchunks):
        """-1 auto, 1 off, n > 1: calibrate in n element chunks on n streams (small graphs)."""
        self.lib.check(self.lib.pgbp_batch_set_pipeline(self.handle, int(nchunks)))

    def set_tilewalk_mode(self, mode):
        """-1 auto, 0 off, 1 on: one launch per traversal for deep schedules of tiny messages."""
        self.lib.check(self.lib.pgbp_batch_set_tilewalk_mode(self.handle, int(mode)))

    def set_tilewalk_params(self, lanes=0, wide=0):
        """message lanes per block (4 / 8 / 16) and the step width launched on its own; 0 = unchanged."""
        self.lib.check(self.lib.pgbp_batch_set_tilewalk_params(self.handle, int(lanes), int(wide)))

    def set_graph_mode(self, mode):
        """-1 auto, 0 off, 1 on: CUDA-graph capture / replay of calibrate calls."""
        self.lib.check(self.lib.pgbp_batch_set_graph_mode(self.handle, int(mode)))

    def set_coop_mode(self, mode):
        """-1 auto, 1 shared-memory kernel, 4 / 8 cooperative lanes, 0 thread-local generic kernel."""
        self.lib.check(self.lib.pgbp_batch_set_coop_mode(self.handle, int(mode)))

    def synchronize(self):
        self.lib.check(self.lib.pgbp_batch_synchronize(self.handle))

    # -- belief access (1-based belief index j) ----------------------------
    def set_belief(self, j, J=None, h=None, g=None):
        m = self.dimension(j)
        # numpy (B,m,m) C-order with J symmetric == Julia (m,m,B) column-major
        Ja = None if J is None else np.ascontiguousarray(np.broadcast_to(np.asarray(J, float), (self.B, m, m)).transpose(0, 2, 1))
        ha = None if h is None else np.ascontiguousarray(np.broadcast_to(np.asarray(h, float), (self.B, m)))
        ga = None if g is None else np.ascontiguousarray(np.broadcast_to(np.asarray(g, float), (self.B,)))
        self.lib.check(self.lib.pgbp_set_belief(self.handle, j - 1, _fptr(Ja), _fptr(ha), _fptr(ga)))

    def _get(self, fn, j, m):
        J = np.empty((self.B, m, m)); h = np.empty((self.B, m)); g = np.empty(self.B)
        self.lib.check(fn(self.handle, j - 1, _fptr(J), _fptr(h), _fptr(g)))
        return J.transpose(0, 2, 1), h, g

    def get_belief(self, j):
        """(J[B,m,m], h[B,m], g[B]) of belief j."""
        return self._get(self.lib.pgbp_get_belief, j, self.dimension(j))

    def get_factor(self, j):
        return self._get(self.lib.pgbp_get_factor, j, self.dimension(j))

    def get_residual(self, sepset_j, to_cluster):
        """MessageResidual of the message into cluster `to_cluster` through
        sepset belief `sepset_j` (both 1-based belief indices)."""
        s = self.dimension(sepset_j)
        dJ = np.empty((self.B, s, s)); dh = np.empty((self.B, s)); fl = np.empty(self.B, dtype=np.uint8); kl = np.empty(self.B)
        self.lib.check(self.lib.pgbp_get_residual(self.handle, sepset_j - 1 - self.nclusters, to_cluster - 1, _fptr(dJ),
                                                  _fptr(dh), fl.ctypes.data_as(C.POINTER(C.c_uint8)), _fptr(kl)))
        return dJ.transpose(0, 2, 1), dh, fl.astype(bool), kl

    def status(self):
        st = np.empty(self.B, dtype=np.int32)
        self.lib.check(self.lib.pgbp_get_status(self.handle, st.ctypes.data_as(_i32p)))
        return st

    def clear_status(self):
        self.lib.check(self.lib.pgbp_clear_status(self.handle))

    # -- initialisation ------------------------------------------------------
    def assignfactors(self, params, tipdata=None, ncolors=1, pairing="zip"):
        """assignfactors! for Brownian-motion models, on the device.  params:
        (nparamsets, len) from bm_params; tipdata: (ndatasets, ntips, ntraits)."""
        pa = np.ascontiguousarray(np.atleast_2d(np.asarray(params, dtype=float)))
        td = None
        nd = 1
        if tipdata is not None:
            td = np.asarray(tipdata, dtype=float)
            if td.ndim == 2:
                td = td[None]
            # (missing data = NaN is not handled by the device path: such elements get a non-zero status from
            # the kernel, status word PGBP_STATUS(0x7ffffa, trait), instead of a host-side scan of the table)
            td = np.ascontiguousarray(td)
            nd = td.shape[0]
        pr = {"zip": L.PAIR_ZIP, "product": L.PAIR_PRODUCT}[pairing]
        self.lib.check(self.lib.pgbp_assign_factors(self.handle, int(ncolors), _fptr(pa), pa.shape[0], _fptr(td), nd, pr))

    init_factors_frommodel = assignfactors

    def assignfactors_ou(self, params, tipdata, pairing="zip"):
        """assignfactors! for UnivariateOrnsteinUhlenbeck on the device.  params: (nparamsets, 5) records
        (sigma2, alpha, theta, mu, v) with v = 0 fixed root, inf improper; tipdata: (ndatasets, ntips, 1)."""
        pa = np.ascontiguousarray(np.atleast_2d(np.asarray(params, dtype=float)))
        if pa.shape[1] != 5:
            raise ValueError("OU parameter records are (sigma2, alpha, theta, mu, v)")
        td = np.asarray(tipdata, dtype=float)
        if td.ndim == 2:
            td = td[None]
        td = np.ascontiguousarray(td)
        pr = {"zip": L.PAIR_ZIP, "product": L.PAIR_PRODUCT}[pairing]
        self.lib.check(self.lib.pgbp_assign_factors_ou(self.handle, _fptr(pa), pa.shape[0], _fptr(td), td.shape[0], pr))

    def assignfactors_device(self, d_params_ptr, nparamsets, d_tip_ptr, ndatasets, ncolors=1, pairing="zip"):
        """assignfactors! with the parameter / tip-data records already on the device (enqueue only)."""
        pr = {"zip": L.PAIR_ZIP, "product": L.PAIR_PRODUCT}[pairing]
        self.lib.check(self.lib.pgbp_assign_factors_device(
            self.handle, int(ncolors), C.c_void_p(int(d_params_ptr)), int(nparamsets),
            C.c_void_p(int(d_tip_ptr)) if d_tip_ptr else None, int(ndatasets), pr))

    def _mem_parent(self):
        if getattr(self, "_mp", None) is None:  # the family table is static: converted once per batch
            fam = self.plan.families
            if fam is None or fam.get("mem_parent") is None:
                raise ValueError("simulate needs the key 'mem_parent' in the plan's node-family table (plan.families)")
            self._mp = _ia(fam["mem_parent"])
        return self._mp

    def simulate(self, params, seed, first_replicate=0, model="bm", ncolors=1, nodes=False):
        """Trait replicates simulated down the network on the device (pgbp_simulate): element e is replicate
        first_replicate + e of `seed`.  params: (nparamsets, len) records of bm_params (model="bm") or (sigma2, alpha,
        theta, mu, v) (model="ou"), nparamsets in {1, B}.  Returns tipdata[B, ntips, p] (NaN where the plan's tip is
        missing), and nodes[B, nnodes, p] (every node, preorder) when nodes=True."""
        mp = self._mem_parent()
        pa = np.ascontiguousarray(np.atleast_2d(np.asarray(params, dtype=float)))
        fam, p = self.plan.families, self.plan.ntraits
        tip = np.empty((self.B, int(fam["ntips"]), p))
        nd = np.empty((self.B, int(fam["nnodes"]), p)) if nodes else None
        self.lib.check(self.lib.pgbp_simulate(self.handle, {"bm": L.MODEL_BM, "ou": L.MODEL_OU}[model], int(ncolors),
                                              mp[1], _fptr(pa), pa.shape[0], int(np.int64(np.uint64(seed))),
                                              int(first_replicate), _fptr(tip), _fptr(nd)))
        return (tip, nd) if nodes else tip

    def simulate_device(self, d_params_ptr, nparamsets, seed, d_tip_ptr, d_nodes_ptr=None, first_replicate=0,
                        model="bm", ncolors=1):
        """simulate with device records and outputs (d_tip [B][ntips][p], d_nodes [B][nnodes][p]; either may be
        None, not both), enqueue only."""
        mp = self._mem_parent()
        self.lib.check(self.lib.pgbp_simulate_device(
            self.handle, {"bm": L.MODEL_BM, "ou": L.MODEL_OU}[model], int(ncolors), mp[1], C.c_void_p(int(d_params_ptr)),
            int(nparamsets), int(np.int64(np.uint64(seed))), int(first_replicate),
            C.c_void_p(int(d_tip_ptr)) if d_tip_ptr else None, C.c_void_p(int(d_nodes_ptr)) if d_nodes_ptr else None))

    def init_beliefs_reset(self):
        self.lib.check(self.lib.pgbp_reset_beliefs(self.handle))

    def init_factors_frombeliefs(self):
        self.lib.check(self.lib.pgbp_factors_from_beliefs(self.handle))

    def init_beliefs_reset_fromfactors(self):
        self.lib.check(self.lib.pgbp_reset_from_factors(self.handle))

    def init_messagecalibrationflags_reset(self, reset_kl=True):
        self.lib.check(self.lib.pgbp_reset_calibration_flags(self.handle, int(reset_kl)))

    # -- message passing -------------------------------------------------------
    def _flags(self, update_residualnorm, update_residualkldiv, auto, reference_order=False):
        f = L.CAL_REFORDER if reference_order else 0
        if update_residualnorm:
            f |= L.CAL_RESIDNORM
        if update_residualkldiv:
            f |= L.CAL_RESIDKLDIV
        if auto:
            f |= L.CAL_AUTO
        return f

    def calibrate(self, schedule=None, niter=1, auto=False, info=False, verbose=True,
                  update_residualnorm=True, update_residualkldiv=False, direction=L.CAL_BOTH, reference_order=False):
        """calibrate!(beliefs, schedule, niter; ...) -> (succ[B], iscal[B])
        [, iter_tree[B,2] if info].  reference_order=True: validation mode PGBP_CAL_REFORDER (every message in the
        reference's LAPACK-style operation order; slow)."""
        ids = None if schedule is None else [self.plan.tree_id(s) for s in schedule]
        ida, idp = (None, None) if ids is None else _ia(ids)
        succ = np.zeros(self.B, dtype=np.int32); iscal = np.zeros(self.B, dtype=np.int32)
        it = np.zeros((self.B, 2), dtype=np.int32) if info else None
        self.lib.check(self.lib.pgbp_calibrate(
            self.handle, idp, 0 if ids is None else len(ids), int(niter),
            direction | self._flags(update_residualnorm, update_residualkldiv, auto, reference_order),
            succ.ctypes.data_as(_i32p), iscal.ctypes.data_as(_i32p), None if it is None else it.ctypes.data_as(_i32p)))
        if info:
            return succ.astype(bool), iscal.astype(bool), it
        return succ.astype(bool), iscal.astype(bool)

    def calibrate_async(self, schedule=None, niter=1, auto=False, update_residualnorm=True, direction=L.CAL_BOTH):
        ids = None if schedule is None else [self.plan.tree_id(s) for s in schedule]
        ida, idp = (None, None) if ids is None else _ia(ids)
        self.lib.check(self.lib.pgbp_calibrate_async(self.handle, idp, 0 if ids is None else len(ids), int(niter),
                                                     direction | self._flags(update_residualnorm, False, auto)))

    def propagate_1traversal_postorder(self, spt, verbose=True, update_residualnorm=True, update_residualkldiv=False):
        """-> succ[B] (src/calibration.jl:111-135)."""
        return self.calibrate([spt], 1, update_residualnorm=update_residualnorm,
                              update_residualkldiv=update_residualkldiv, direction=L.CAL_POSTORDER)[0]

    def propagate_1traversal_preorder(self, spt, verbose=True, update_residualnorm=True, update_residualkldiv=False):
        return self.calibrate([spt], 1, update_residualnorm=update_residualnorm,
                              update_residualkldiv=update_residualkldiv, direction=L.CAL_PREORDER)[0]

    def propagate_belief(self, to, sepset, frm):
        """propagate_belief!(cluster_to, sepset, cluster_from, residual) with
        1-based belief indices; failures are recorded in status()."""
        self.lib.check(self.lib.pgbp_propagate(self.handle, frm - 1, sepset - 1, to - 1, 0))

    def integratebelief(self, j, want_mu=True):
        """integratebelief!(beliefs, j) -> (mu[B,m], norm[B])."""
        m = self.dimension(j)
        mu = np.empty((self.B, m)) if want_mu else None
        norm = np.empty(self.B)
        self.lib.check(self.lib.pgbp_integrate(self.handle, j - 1, _fptr(mu), _fptr(norm)))
        return mu, norm

    def integratebelief_cov(self, j):
        """integratebelief!(beliefs, j) + inv(J) -> (mu[B,m], cov[B,m,m], norm[B]): the conditional moments
        used by calibrate_exact_cliquetree! (src/calibration.jl:462-463)."""
        m = self.dimension(j)
        mu = np.empty((self.B, m)); cov = np.empty((self.B, m, m)); norm = np.empty(self.B)
        self.lib.check(self.lib.pgbp_integrate_cov(self.handle, j - 1, _fptr(mu), _fptr(cov), _fptr(norm)))
        return mu, cov, norm

    @staticmethod
    def _query_arrays(queries):
        qb, off, pos = [], [0], []
        for j, p in queries:
            qb.append(int(j) - 1)
            pos.extend(int(x) for x in p)
            off.append(len(pos))
        return _ia(qb), _ia(off), _ia(pos or [0]), off

    def marginal_moments(self, queries):
        """Posterior moments of position subsets of beliefs (pgbp_marginal_moments): `queries` is a list of
        (belief_j, positions), 1-based belief index, 0-based positions in its scope.  Returns one (mu[B,k], cov[B,k,k])
        per query -- mu = (J^-1 h)[pos], cov = inv(J)[pos, pos], bit-identical to those entries of
        integratebelief_cov -- as views into one packed result.  Each belief is factorised once however many queries
        name it.  All-zero belief: +Inf; J not positive definite: NaN and a status word for that element."""
        (qa, qp), (oa, op), (pa, pp), off = self._query_arrays(queries)
        ks = np.diff(off)
        mu = np.empty((self.B, int(ks.sum())))
        cov = np.empty((self.B, int((ks * ks).sum())))
        self.lib.check(self.lib.pgbp_marginal_moments(self.handle, len(ks), qp, op, pp, _fptr(mu), _fptr(cov)))
        out, m0, c0 = [], 0, 0
        for k in ks:
            k = int(k)
            # column-major k x k per query
            out.append((mu[:, m0:m0 + k], cov[:, c0:c0 + k * k].reshape(self.B, k, k).transpose(0, 2, 1)))
            m0 += k
            c0 += k * k
        return out

    def marginal_moments_device(self, queries, d_mu_ptr, d_cov_ptr=None):
        """pgbp_marginal_moments_device, enqueue only: query q's mean into rows [sum_{q'<q} k_q' ...) of the device
        array d_mu ([sum k][ld] doubles, ld of device_view()), its packed upper covariance triangle into rows
        [sum_{q'<q} k_q'(k_q'+1)/2 ...) of d_cov ([sum k(k+1)/2][ld]); d_cov may be None."""
        (qa, qp), (oa, op), (pa, pp), off = self._query_arrays(queries)
        self.lib.check(self.lib.pgbp_marginal_moments_device(self.handle, len(off) - 1, qp, op, pp,
                                                             C.c_void_p(int(d_mu_ptr)),
                                                             C.c_void_p(int(d_cov_ptr)) if d_cov_ptr else None))

    def node_queries(self):
        """The node-family table's query of every network node with a trait in scope: [(v, traits, belief_j,
        positions)] with v the 0-based preorder node index, `traits` its in-scope traits (0-based), belief_j its home
        cluster node_cluster[v] (1-based) and `positions` those traits' positions in the cluster's scope (its own
        member entry: mem_pos + t, or mem_tpos with partial scopes)."""
        if getattr(self, "_node_queries", None) is not None:  # the family table is static: computed once per batch
            return self._node_queries
        fam = self.plan.families
        if fam is None:
            raise ValueError("node moments need the plan's node-family table (ClusterGraphPlan(families=...))")
        p = self.plan.ntraits
        tpos = fam.get("mem_tpos")
        out = []
        for v in range(int(fam["nnodes"])):
            a = fam["mem_off"][v]  # the node's own member entry (members are listed child first)
            if tpos is not None:
                tp = [int(tpos[a * p + t]) for t in range(p)]
            else:
                base = int(fam["mem_pos"][a])
                tp = [base + t if base >= 0 else -1 for t in range(p)]
            traits = [t for t in range(p) if tp[t] >= 0]
            if traits:
                out.append((v, traits, int(fam["node_cluster"][v]) + 1, [tp[t] for t in traits]))
        self._node_queries = out
        return out

    def node_moments(self):
        """Posterior distribution of every network node given the data (ancestral state reconstruction):
        (mu[B, nnodes, p], cov[B, nnodes, p, p], in_scope[nnodes, p]) from each node's home cluster (node_queries).
        Traits out of scope are NaN (in mu and in their covariance rows and columns): every trait of a tip (observed
        values are evidence, missing ones are integrated out of the tip's edge factor, src/beliefs.jl:833-857), a
        trait with no data below an internal node, a fixed root.  On a loopy cluster graph the result is the home cluster's
        approximate (belief-propagation) marginal."""
        nq = self.node_queries()
        n, p = int(self.plan.families["nnodes"]), self.plan.ntraits
        mu = np.full((self.B, n, p), np.nan)
        cov = np.full((self.B, n, p, p), np.nan)
        ins = np.zeros((n, p), dtype=bool)
        if nq:
            res = self.marginal_moments([(j, pos) for _, _, j, pos in nq])
            for (v, tr, _, _), (m, c) in zip(nq, res):
                t = np.asarray(tr)
                ins[v, t] = True
                mu[:, v, t] = m
                cv = cov[:, v]
                cv[:, t[:, None], t[None, :]] = c
        return mu, cov, ins

    def node_moments_device(self, d_mu_ptr, d_cov_ptr=None):
        """node_moments into device arrays, enqueue only: the rows are those of marginal_moments_device for the
        queries of node_queries(), in that order (sum of in-scope traits rows of d_mu, sum k(k+1)/2 of d_cov)."""
        nq = self.node_queries()
        if not nq:
            raise ValueError("no network node has a trait in scope")
        self.marginal_moments_device([(j, pos) for _, _, j, pos in nq], d_mu_ptr, d_cov_ptr)

    def factored_energy(self):
        """-> [B,3] = (average energy, approximate entropy, factored energy)."""
        out = np.empty((self.B, 3))
        self.lib.check(self.lib.pgbp_factored_energy(self.handle, _fptr(out)))
        return out

    def free_energy(self):
        fe = self.factored_energy()
        fe[:, 2] = -fe[:, 2]
        return fe

    # -- regularisation ------------------------------------------------------------
    def regularizebeliefs_bycluster(self):
        self.lib.check(self.lib.pgbp_regularize_bycluster(self.handle))

    def regularizebeliefs_onschedule(self):
        self.lib.check(self.lib.pgbp_regularize_onschedule(self.handle))

    def regularizebeliefs_bynodesubtree(self, program):
        """program: list of (eps_clusters, [(cluster, sepset_belief, c_ind, s_ind)])
        per network node, 1-based belief indices, 0-based diagonal positions --
        the loop body of src/clustergraphbeliefs.jl:314-340 as index data."""
        eo, ec, so, sc, ss, io, ic, is_ = [0], [], [0], [], [], [0], [], []
        for epscl, steps in program:
            ec.extend(c - 1 for c in epscl); eo.append(len(ec))
            for ci, si, c_ind, s_ind in steps:
                sc.append(ci - 1); ss.append(si - 1 - self.nclusters)
                ic.extend(int(x) for x in c_ind); is_.extend(int(x) for x in s_ind); io.append(len(ic))
            so.append(len(sc))
        arrs = [_ia(x or [0]) for x in (eo, ec, so, sc, ss, io, ic, is_)]
        self.lib.check(self.lib.pgbp_regularize_bynodesubtree(self.handle, len(program), *[a[1] for a in arrs]))

    # -- device views ----------------------------------------------------------------
    def device_view(self):
        base, ld, ns = C.c_void_p(), C.c_int64(), C.c_int64()
        self.lib.check(self.lib.pgbp_device_view(self.handle, C.byref(base), C.byref(ld), C.byref(ns)))
        return base.value, ld.value, ns.value

    def factored_energy_device(self, d_out_ptr):
        """factored_energy into a device array [3][ld] (energy, entropy, factored energy), enqueue only."""
        self.lib.check(self.lib.pgbp_factored_energy_device(self.handle, C.c_void_p(int(d_out_ptr))))

    def integrate_device(self, j, d_norm_ptr, d_mu_ptr=None):
        self.lib.check(self.lib.pgbp_integrate_device(self.handle, j - 1, C.c_void_p(d_mu_ptr) if d_mu_ptr else None,
                                                      C.c_void_p(int(d_norm_ptr))))


# reference-style free functions -------------------------------------------------------
def calibrate(beliefs, schedule, niter=1, **kw):
    return beliefs.calibrate(schedule, niter, **kw)


def propagate_1traversal_postorder(beliefs, spt, *a, **kw):
    return beliefs.propagate_1traversal_postorder(spt, *a, **kw)


def propagate_1traversal_preorder(beliefs, spt, *a, **kw):
    return beliefs.propagate_1traversal_preorder(spt, *a, **kw)


def propagate_belief(beliefs, to, sepset, frm):
    return beliefs.propagate_belief(to, sepset, frm)


def integratebelief(beliefs, j, **kw):
    return beliefs.integratebelief(j, **kw)


def factored_energy(beliefs):
    return beliefs.factored_energy()


def free_energy(beliefs):
    return beliefs.free_energy()


def regularizebeliefs_bycluster(beliefs, cgraph=None):
    return beliefs.regularizebeliefs_bycluster()


def regularizebeliefs_onschedule(beliefs, cgraph=None):
    return beliefs.regularizebeliefs_onschedule()


def regularizebeliefs_bynodesubtree(beliefs, program):
    return beliefs.regularizebeliefs_bynodesubtree(program)


def init_beliefs_reset_fromfactors(beliefs):
    return beliefs.init_beliefs_reset_fromfactors()


def init_factors_frombeliefs(beliefs):
    return beliefs.init_factors_frombeliefs()


def init_messagecalibrationflags_reset(beliefs, reset_kl=True):
    return beliefs.init_messagecalibrationflags_reset(reset_kl)


def assignfactors(beliefs, params, tipdata=None, **kw):
    return beliefs.assignfactors(params, tipdata, **kw)


init_factors_frommodel = assignfactors
