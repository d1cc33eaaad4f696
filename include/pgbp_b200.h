/*
 * libpgbp_b200 -- C ABI of the B200-native Gaussian belief-propagation library.
 *
 * Drop-in boundary for the message-passing hot path of
 * JuliaPhylo/PhyloGaussianBeliefProp.jl (reference paths below are relative to
 * that checkout).  The reference has no FFI of its own: the path sits behind
 * ordinary Julia functions on `ClusterGraphBelief`; each entry point here is
 * what a thin `ccall` method of the same Julia name binds to (INTEGRATION.md
 * shows the Julia side).  Batched: one call processes B independent
 * (J,h,g) replicas of the same cluster graph (trait replicates and/or
 * parameter vectors).
 *
 * Conventions
 *  - every function returns int32: 0 = ok, <0 = API misuse / CUDA error
 *    (text via pgbp_last_error).  Nothing throws across the ABI.
 *  - numerical failure is NOT an error code.  Like the reference's
 *    propagate_belief!, which RETURNS its BPPosDefException instead of
 *    throwing (src/beliefupdates.jl:640-644), a failed Cholesky is recorded
 *    per batch element in status[e] (0 = ok, else PGBP_STATUS(message, pivot))
 *    and that element stops updating; the rest of the batch is unaffected.
 *  - all indices are 0-based int32; all reals are IEEE binary64.
 *  - host matrices are dense column-major m x m per element, element-major
 *    across the batch, so a Julia Array{Float64,3} of size (m,m,B) (resp.
 *    (m,B) for vectors, (B,) for scalars) maps directly.
 *  - caller owns every host buffer for the duration of the call (Julia:
 *    GC.@preserve); the library owns device memory (freed by *_destroy).
 *  - a pgbp_batch is bound to one device and one stream; calls on one batch
 *    are not re-entrant; distinct batches may be driven from distinct host
 *    threads.  Calls taking host pointers are synchronous at return; the
 *    *_device variants only enqueue work on the batch's stream.
 */
#ifndef PGBP_B200_H
#define PGBP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PGBP_ABI_VERSION 2

typedef struct pgbp_plan pgbp_plan;
typedef struct pgbp_batch pgbp_batch;

/* status word of a failed element: message id is the 0-based position of the
 * failing message in the reference's sequential order for that call (post-order
 * messages first, then pre-order, per tree, per iteration); pivot is LAPACK's
 * 1-based `info` (BPPosDefException.info, src/beliefupdates.jl:11-14). */
#define PGBP_STATUS(msg, pivot) ((int32_t)((((uint32_t)(msg) + 1u) << 8) | ((uint32_t)(pivot) & 0xffu)))
#define PGBP_STATUS_MSG(st) ((int32_t)(((uint32_t)(st)) >> 8) - 1)
#define PGBP_STATUS_PIVOT(st) ((int32_t)((st) & 0xff))

/* ---------------------------------------------------------------- node families
 * Optional table for pgbp_assign_factors (replaces assignfactors!,
 * src/beliefs.jl:786-861, for Brownian-motion models without missing data).
 * Node v = 0-based preorder index.  Members of family v are listed child first,
 * then parents by decreasing preorder index (src/beliefs.jl:515-524,535). */
typedef struct pgbp_family_table {
  int32_t nnodes;              /* network nodes */
  int32_t ntips;               /* rows of a tip-data set */
  const int32_t* node_cluster; /* [nnodes] cluster holding family v (node2cluster) */
  const int32_t* mem_off;      /* [nnodes+1] offsets into mem_* (1 + #parents entries per node) */
  const int32_t* mem_pos;      /* position of the member's first variable inside that cluster's
                                  scope (scopeindex, src/beliefs.jl:354-373), -1 if the member is
                                  fixed (a tip with data, or a fixed root) */
  const double* mem_length;    /* parent-edge length t_k   (entry of the child itself: unused) */
  const double* mem_gamma;     /* inheritance gamma_k      (1 for tree edges) */
  const int32_t* mem_color;    /* rate colour of the parent edge (PaintedParameter,
                                  src/evomodels/heterogeneousmodels.jl:21-33), 0 if homogeneous */
  const int32_t* node_datarow; /* [nnodes] row of the tip in the data set, -1 for internal nodes */
  int32_t root_fixed;          /* 1 if the plan was allocated for a fixed root (isrootfixed,
                                  src/evomodels/evomodels.jl:41): the root is out of scope */
  /* Trait-level scopes (missing data; src/beliefs.jl:505-559, 833-857).  Both NULL = every non-fixed
   * member has all its traits in scope and no tip value is missing (the fast paths). */
  const int32_t* mem_tpos;     /* [#members * ntraits] position of trait t of the member inside the
                                  cluster's scope, -1 if that trait is out of scope (all -1 for a
                                  fixed member); when given, mem_pos only says whether the member is
                                  fixed (< 0) or not (>= 0) */
  const uint8_t* tip_missing;  /* [ntips * ntraits] 1 = this trait is missing at this tip in every data
                                  set (the pattern the beliefs were allocated for); those entries of
                                  `tipdata` are not read */
} pgbp_family_table;

/* ---------------------------------------------------------------- plan
 * Everything static about one cluster graph: belief dimensions, the
 * (sepset, cluster) scope maps and the message schedules.  It is the output of
 * the reference's graph layer, consumed as is:
 *   belief order  = clusters in labels(cgraph) order, then sepsets in
 *                   edge_labels(cgraph) order        (src/beliefs.jl:561-592)
 *   upind         = scopeindex(sepset, cluster)      (src/beliefs.jl:389-405)
 *   tree k        = spanningtree_clusterlist output  (src/clustergraph.jl:881-894):
 *                   edges in preorder, parent/child cluster indices. */
typedef struct pgbp_plan_desc {
  int32_t nclusters;
  int32_t nsepsets;
  int32_t ntraits;
  const int32_t* belief_dim;      /* [nclusters+nsepsets] */
  const int32_t* sepset_clusters; /* [2*nsepsets] (cluster_a, cluster_b) = metadata order */
  const int32_t* upind_off;       /* [2*nsepsets+1] */
  const int32_t* upind;           /* scope of sepset j inside cluster_a: upind[upind_off[2j]..),
                                     inside cluster_b: upind[upind_off[2j+1]..); ascending */
  int32_t ntrees;
  const int32_t* tree_off;        /* [ntrees+1] */
  const int32_t* tree_parent;     /* concatenated parent cluster indices */
  const int32_t* tree_child;      /* concatenated child cluster indices  */
  const pgbp_family_table* families; /* NULL if pgbp_assign_factors is not used */
} pgbp_plan_desc;

int32_t pgbp_abi_version(void);
int32_t pgbp_last_error(char* buf, size_t buflen);

int32_t pgbp_plan_create(const pgbp_plan_desc* desc, pgbp_plan** out);
int32_t pgbp_plan_destroy(pgbp_plan* plan);

/* Flattened schedule, for diffing against the host mirror.  A traversal
 * (direction 0 = postorder child->parent, 1 = preorder parent->child) of tree
 * `tree` is cut into launch steps; messages inside one step are independent
 * and have distinct receivers; steps run in order.  Out arrays have one entry
 * per message of the traversal (tree size), in execution order:
 *   msg_ref[i]   position of the message in the reference's sequential order
 *                (src/calibration.jl:121,147)
 *   msg_step[i]  step it runs in
 *   msg_from/msg_sepset/msg_to[i]  belief indices (sepset = nclusters + j)
 * Pass NULL arrays to query *nmsg / *nsteps only. */
int32_t pgbp_plan_get_levels(const pgbp_plan* plan, int32_t tree, int32_t direction,
                             int32_t* nmsg, int32_t* nsteps, int32_t* msg_ref, int32_t* msg_step,
                             int32_t* msg_from, int32_t* msg_sepset, int32_t* msg_to);

/* Algorithmic bytes / flops of one traversal per batch element (SURVEY.md 8d):
 * symmetric-packed beliefs, every element independent. */
int32_t pgbp_plan_traversal_cost(const pgbp_plan* plan, int32_t tree, int32_t direction,
                                 int32_t track_residuals, double* bytes, double* flops);

/* ---------------------------------------------------------------- batch */
#define PGBP_BATCH_FACTORS 1u   /* keep the factor snapshot (needed by factored_energy / reset) */
#define PGBP_BATCH_RESIDUALS 2u /* keep message residuals (needed for iscal / loopy BP) */

int32_t pgbp_batch_create(const pgbp_plan* plan, int64_t B, int32_t device, uint32_t flags,
                          pgbp_batch** out);
/* Shared-precision batch: the `group_size` consecutive elements of a group use ONE parameter vector
 * (trait replicates under one theta), so every J of the group is the same matrix (only h and g depend on
 * the data, src/beliefupdates.jl:77-81).  J is stored ONCE per group (HBM per element: 8 (m+1) bytes per belief
 * instead of 8 (m(m+1)/2 + m + 1)); a message factorises J_I once per group (one warp per (message, group)),
 * caches U, Z = U^-T J_IK and logdet, and every element only applies them to its h and g.  Same calls, same
 * results (bit for bit) as an ordinary batch given the same inputs; restrictions: pgbp_assign_factors needs one
 * parameter set per group, calibrate has no auto-stop (it is per element) and no reference-order mode,
 * pgbp_set_belief takes J from each group's first element, an element whose h_I is non-zero where the group's
 * J_I, J_IK are zero fails (status) instead of taking the reference's data-dependent branch.
 * group_size 0 or 1 = ordinary batch (every element its own J). */
int32_t pgbp_batch_create_shared(const pgbp_plan* plan, int64_t B, int64_t group_size, int32_t device,
                                 uint32_t flags, pgbp_batch** out);
int32_t pgbp_batch_destroy(pgbp_batch* batch);
/* run on an externally owned cudaStream_t (e.g. the caller's current stream) */
int32_t pgbp_batch_set_stream(pgbp_batch* batch, void* cuda_stream);
int32_t pgbp_batch_synchronize(pgbp_batch* batch);
int64_t pgbp_batch_size(const pgbp_batch* batch);
int64_t pgbp_batch_device_bytes(const pgbp_batch* batch);
/* kernels launched on this batch since creation / since the last reset (reset != 0) */
int64_t pgbp_batch_launch_count(pgbp_batch* batch, int32_t reset);

/* Kernel strategy of calibrate / traversals: -1 automatic (default; currently always 0),
 * 0 level-parallel launches (one launch per step and shape class; parallel over messages and
 * replicates), 1 walk kernel (one launch per traversal; each thread walks all messages of its
 * replicate; needs every message shape to be whole nodes of ntraits <= 4 traits, else falls
 * back to 0).  Results are bit-identical. */
int32_t pgbp_batch_set_walk_mode(pgbp_batch* batch, int32_t mode);
/* Pipelined calibration: the batch is cut into `nchunks` ranges of elements; every range walks the
 * whole schedule on its own stream (elements are independent), so the ramp-up and tail of the small
 * launches of one range overlap the other ranges' work.  -1 automatic (default: up to 4 chunks of
 * >= 8192 elements when one launch cannot fill the GPU), 1 off.  Results are unaffected. */
int32_t pgbp_batch_set_pipeline(pgbp_batch* batch, int32_t nchunks);
/* Tile-walk kernel for deep schedules of tiny messages (sender dimension <= 4; loopy BP on Bethe-type
 * graphs): one launch per run of consecutive narrow steps, a block walks the steps for its 32 elements
 * with a block barrier between steps; steps wider than `wide` messages keep their ordinary launches.
 * -1 automatic (default: on for traversals of >= 24 steps averaging < 32 messages), 0 off, 1 on wherever
 * applicable.  Results are unaffected (same per-message arithmetic). */
int32_t pgbp_batch_set_tilewalk_mode(pgbp_batch* batch, int32_t mode);
/* Tuning of the tile-walk kernel: message lanes per block (4, 8 or 16; default 8) and the step width above
 * which a step is launched on its own (default 512).  0 keeps the current value. */
int32_t pgbp_batch_set_tilewalk_params(pgbp_batch* batch, int32_t lanes, int32_t wide);
/* CUDA-graph replay of calibrate calls: -1 automatic (default: calls of >= 24 launches are captured at
 * their second occurrence and replayed afterwards), 0 off, 1 always.  Results are unaffected. */
int32_t pgbp_batch_set_graph_mode(pgbp_batch* batch, int32_t mode);
/* Kernel for medium message shapes (sender dimension > 12): -1 automatic (shared-memory kernel where it
 * fits; integrated dimensions 12..16 use its multi-warp form: 8 warps share one tile of 32 elements and
 * split the work by column), 1 single-warp shared-memory kernel (one thread per element, factor in
 * shared memory), 2 multi-warp form with 4 warps, 4 / 8 cooperative kernel (that many lanes per element
 * for sender dimensions <= 16, 8 above; sender dimension <= 48), 0 one thread per element with
 * thread-local storage.  Results are bit-identical. */
int32_t pgbp_batch_set_coop_mode(pgbp_batch* batch, int32_t mode);

/* Host <-> device belief access (CanonicalBelief fields, src/beliefs.jl:72-132).
 * J: [B][m][m] column-major full square, h: [B][m], g: [B]; any pointer may be
 * NULL.  set symmetrises nothing: the upper triangle is taken, as the
 * reference's Cholesky does (PDMat(Symmetric(J)), src/beliefupdates.jl:68). */
int32_t pgbp_set_belief(pgbp_batch* batch, int32_t belief, const double* J, const double* h,
                        const double* g);
int32_t pgbp_get_belief(pgbp_batch* batch, int32_t belief, double* J, double* h, double* g);
/* ClusterFactor access (src/beliefs.jl:6-16), clusters only */
int32_t pgbp_get_factor(pgbp_batch* batch, int32_t cluster, double* J, double* h, double* g);
/* MessageResidual of the message sent INTO cluster `to` through sepset j
 * (key (label_to,label_from), src/beliefs.jl:895-924): dJ [B][s][s], dh [B][s],
 * iscalibrated_resid [B] (uint8), kldiv [B] */
int32_t pgbp_get_residual(pgbp_batch* batch, int32_t sepset, int32_t to_cluster, double* dJ,
                          double* dh, uint8_t* iscal_resid, double* kldiv);
int32_t pgbp_get_status(pgbp_batch* batch, int32_t* status);
int32_t pgbp_clear_status(pgbp_batch* batch);

/* init_beliefs_reset! (src/beliefs.jl:706-717) */
int32_t pgbp_reset_beliefs(pgbp_batch* batch);
/* init_factors_frombeliefs! (src/beliefs.jl:747-761) */
int32_t pgbp_factors_from_beliefs(pgbp_batch* batch);
/* init_beliefs_reset_fromfactors! (src/clustergraphbeliefs.jl:126-139) */
int32_t pgbp_reset_from_factors(pgbp_batch* batch);
/* init_messagecalibrationflags_reset! (src/clustergraphbeliefs.jl:146-150) */
int32_t pgbp_reset_calibration_flags(pgbp_batch* batch, int32_t reset_kl);

/* ---------------------------------------------------------------- factor assignment
 * assignfactors! (src/beliefs.jl:786-861) fused with the Brownian-motion factor
 * formulas (src/evomodels/homogeneousbrownianmotion.jl:222-351,
 * src/evomodels/heterogeneousmodels.jl:119-150, src/evomodels/evomodels.jl:377-396)
 * and evidence absorption (src/beliefupdates.jl:210-231), then the factor
 * snapshot (src/clustergraphbeliefs.jl:106).  Requires plan.families.  Plans with trait-level
 * scopes (families->mem_tpos / tip_missing: missing data) go through the reference's own sequence --
 * full family factor, absorbleaf!, marginalisation of missing tip traits, fixed-root evidence, two-stage
 * marginalisation of out-of-scope traits (src/beliefs.jl:822-858) -- on the device, one thread per
 * (cluster, element); family size * ntraits <= 48 there.  Other models are assigned on the host and
 * uploaded with pgbp_set_belief + pgbp_factors_from_beliefs.
 *
 * params: nparamsets records of  ncolors*p*p (rates R_c, column-major)
 *                                + p (root mean mu) + p*p (root variance v):
 *         v == 0 fixed root, any diag(v) == Inf improper, else proper prior.
 * tipdata: ndatasets records of ntips*p  (data[row][trait]); a NaN where the plan expects a value
 *          (tip_missing == 0) gives the element the status PGBP_STATUS(0x7ffffa, trait); a failed
 *          marginalisation (src/beliefupdates.jl:68-76) PGBP_STATUS(0x7ffff9, pivot).
 * pairing: element e uses (param, data) = ZIP: (min(e,np-1), min(e,nd-1)) with
 *          np, nd in {1, B};  PRODUCT: (e / nd, e % nd) with np*nd == B. */
#define PGBP_PAIR_ZIP 0
#define PGBP_PAIR_PRODUCT 1
int32_t pgbp_assign_factors(pgbp_batch* batch, int32_t ncolors, const double* params,
                            int64_t nparamsets, const double* tipdata, int64_t ndatasets,
                            int32_t pairing);
/* same with DEVICE pointers (records already in HBM), enqueue only: the optimiser inner loop that
 * keeps its theta grid on the GPU (src/calibration.jl:195-221) */
int32_t pgbp_assign_factors_device(pgbp_batch* batch, int32_t ncolors, const double* d_params,
                                   int64_t nparamsets, const double* d_tipdata, int64_t ndatasets,
                                   int32_t pairing);

/* assignfactors! for the univariate Ornstein-Uhlenbeck model
 * (src/evomodels/homogeneousornsteinuhlenbeck.jl:18-66; generic linear-Gaussian factors of
 * src/evomodels/evomodels.jl:208-245, 314-330).  params: nparamsets records (sigma2, alpha, theta, mu, v),
 * v == 0 fixed root, Inf improper; ntraits must be 1; tipdata / pairing as above. */
int32_t pgbp_assign_factors_ou(pgbp_batch* batch, const double* params, int64_t nparamsets,
                               const double* tipdata, int64_t ndatasets, int32_t pairing);

/* ---------------------------------------------------------------- message passing */
#define PGBP_CAL_POSTORDER 1u       /* propagate_1traversal_postorder! (src/calibration.jl:111-135) */
#define PGBP_CAL_PREORDER 2u        /* propagate_1traversal_preorder!  (src/calibration.jl:137-161) */
#define PGBP_CAL_BOTH 3u            /* calibrate!(beliefs, spt)        (src/calibration.jl:72-84)   */
#define PGBP_CAL_RESIDNORM 4u       /* update_residualnorm  (default true in the reference)  */
#define PGBP_CAL_RESIDKLDIV 8u      /* update_residualkldiv (default false)                  */
#define PGBP_CAL_AUTO 16u           /* auto: an element stops at its first calibrated tree   */
#define PGBP_CAL_REFORDER 32u       /* validation mode: every message in the reference's own operation order (LAPACK-order
                                       upper Cholesky of J_I with division by the pivot, X_invA_Xt accumulated un-fused,
                                       src/beliefupdates.jl:68-81) instead of the fused right-looking form; J and h then
                                       agree bit for bit with a LAPACK-style evaluation of the reference even on
                                       ill-conditioned loopy configurations.  Slow (thread-local kernel); never automatic. */

/* calibrate!(beliefs, schedule, niter; auto, update_residualnorm, update_residualkldiv)
 * (src/calibration.jl:35-60) per element.  tree_ids selects/permutes plan trees
 * (NULL = all, in order).  Outputs (host, may be NULL): succ[B], iscal[B] as in the
 * reference's (succ, iscal) tuple; iter_tree[2B] = 1-based (iteration, tree) at which
 * calibration was first detected, (0,0) if never (the `info` log line). */
int32_t pgbp_calibrate(pgbp_batch* batch, const int32_t* tree_ids, int32_t ntrees, int32_t niter,
                       uint32_t flags, int32_t* succ, int32_t* iscal, int32_t* iter_tree);
/* same, enqueue only (no outputs, no synchronisation) */
int32_t pgbp_calibrate_async(pgbp_batch* batch, const int32_t* tree_ids, int32_t ntrees,
                             int32_t niter, uint32_t flags);

/* propagate_belief!(cluster_to, sepset, cluster_from, residual) (src/beliefupdates.jl:634-665) */
int32_t pgbp_propagate(pgbp_batch* batch, int32_t from_cluster, int32_t sepset, int32_t to_cluster,
                       uint32_t flags);

/* integratebelief!(beliefs, j) (src/clustergraphbeliefs.jl:194, src/beliefupdates.jl:168-200):
 * mu [B][m] (may be NULL), norm [B].  Elements whose Cholesky fails get NaN and a status. */
int32_t pgbp_integrate(pgbp_batch* batch, int32_t belief, double* mu, double* norm);
int32_t pgbp_integrate_device(pgbp_batch* batch, int32_t belief, double* d_mu_soa, double* d_norm);
/* same + the conditional covariance inv(J): cov [B][m][m] -- the moments calibrate_exact_cliquetree!
 * takes from every cluster (integratebelief! + inv(b.J), src/calibration.jl:462-463) */
int32_t pgbp_integrate_cov(pgbp_batch* batch, int32_t belief, double* mu, double* cov, double* norm);

/* Posterior (conditional) moments of variable subsets -- ancestral state reconstruction.  Query q is the marginal
 * Gaussian of belief q_belief[q] on its scope positions q_pos[q_off[q] .. q_off[q+1]) (k_q distinct positions in
 * [0, m), any order): mu = (J^-1 h)[pos] and cov = (J^-1)[pos, pos], i.e. integratebelief!
 * (src/beliefupdates.jl:168-200) + inv(J) restricted to the subset, the node moments the reference reads in
 * test/test_calibration.jl:47-105 and test/test_exactBM.jl:20-52.  Each belief is factorised once per element
 * however many queries name it; entries are bit-identical to the same entries of pgbp_integrate_cov.  On a loopy
 * graph the result is the belief's approximate marginal.  Sepset beliefs are allowed.
 * mu [B][sum k_q] and cov [B][sum k_q^2] (column-major k_q x k_q per query, queries in order); cov may be NULL.
 * Per element: J not positive definite -> status PGBP_STATUS(0x7ffffe, pivot) and NaN in every output of that
 * belief; all-zero (J, h) -> +Inf in every mean and covariance output of that belief (integratebelief's mean;
 * pgbp_integrate_cov leaves its covariance undefined there).
 * PGBP_EINVAL: nq < 1, a null required pointer, a belief out of range, q_off decreasing, a position outside [0, m)
 * or repeated within a query, or (host variant) more than 65535*32 mean or covariance columns. */
int32_t pgbp_marginal_moments(pgbp_batch* batch, int32_t nq, const int32_t* q_belief, const int32_t* q_off,
                              const int32_t* q_pos, double* mu, double* cov);
/* same into device SoA arrays, enqueue only: d_mu rows [sum k_q][ld], d_cov rows [sum k_q(k_q+1)/2][ld] (query q's
 * packed upper triangle, (r <= c) -> c(c+1)/2 + r, after those of queries < q; the layout of pgbp_device_view);
 * d_cov may be NULL */
int32_t pgbp_marginal_moments_device(pgbp_batch* batch, int32_t nq, const int32_t* q_belief, const int32_t* q_off,
                                     const int32_t* q_pos, double* d_mu, double* d_cov);

/* factored_energy (src/score.jl:151-154,162-182): out [B][3] =
 * (average energy, approximate entropy, factored energy) */
int32_t pgbp_factored_energy(pgbp_batch* batch, double* out);
int32_t pgbp_factored_energy_device(pgbp_batch* batch, double* d_out_soa);

/* ---------------------------------------------------------------- regularisation */
/* regularizebeliefs_bycluster! (src/clustergraphbeliefs.jl:235-249) */
int32_t pgbp_regularize_bycluster(pgbp_batch* batch);
/* regularizebeliefs_onschedule! (src/clustergraphbeliefs.jl:376-403) */
int32_t pgbp_regularize_onschedule(pgbp_batch* batch);
/* regularizebeliefs_bynodesubtree! (src/clustergraphbeliefs.jl:306-340).  The host passes the
 * index program of that loop, one record per network node in the order it is to be visited:
 *   eps_off[n..n+1)  -> eps_cluster[]: clusters whose max|J| defines that node's epsilon
 *   step_off[n..n+1) -> (step_cluster, step_sepset)[]: child cluster + sepset along the subtree
 *   idx_off[k..k+1)  -> (idx_cluster, idx_sepset)[]: diagonal positions (scopeindex(node,
 *                       sepset, cluster), src/beliefs.jl:418-436) of step k */
int32_t pgbp_regularize_bynodesubtree(pgbp_batch* batch, int32_t nnodes, const int32_t* eps_off,
                                      const int32_t* eps_cluster, const int32_t* step_off,
                                      const int32_t* step_cluster, const int32_t* step_sepset,
                                      const int32_t* idx_off, const int32_t* idx_cluster,
                                      const int32_t* idx_sepset);

/* ---------------------------------------------------------------- device views (zero-copy)
 * Raw device pointers into the batch's structure-of-arrays state, for callers that
 * keep data on the GPU (e.g. gather of per-replicate log-likelihoods with NCCL).
 * Layout: slot k of element e at base[k * ld + e]; a belief occupies
 * S(m)=m(m+1)/2 slots of J (packed upper, column-major: (r<=c) -> c(c+1)/2 + r),
 * then m slots of h, then 1 slot of g. */
int32_t pgbp_device_view(pgbp_batch* batch, double** base, int64_t* ld, int64_t* nslots);
int32_t pgbp_belief_slot(const pgbp_plan* plan, int32_t belief, int64_t* jslot, int64_t* hslot,
                         int64_t* gslot);
/* Rows of belief i's h (m rows from *hrow) and g (*grow) in the array pgbp_device_view returns.  Ordinary batches:
 * the plan's slots.  Shared-precision batches: that array holds h and g only, in compact rows (the J rows live
 * once per group in an internal group batch). */
int32_t pgbp_batch_belief_rows(const pgbp_batch* batch, int32_t belief, int64_t* hrow, int64_t* grow);

/* ---------------------------------------------------------------- multi-GPU gather over NVLink peer memory
 * The path shards by batch element (one process per GPU, the plan replicated); its only exchange is the gather
 * of the per-replicate results (log-likelihoods), the role of the closing `Threads.@threads` join + result
 * vector of the reference's replicate loop.  Instead of a collective launch per step the exchange is fused into
 * the producing kernel: every rank owns a window of `nbuffers` x `nranks` rows of `ld` doubles, exported with CUDA
 * IPC; after pgbp_comm_connect each rank's integratebelief! kernel stores its results into row `rank` of EVERY
 * rank's window through the peer mappings and publishes a sequence number; pgbp_comm_wait enqueues a wait (on the
 * batch's stream) until all ranks' rows of a buffer have landed.  Handles are 64 opaque bytes the host exchanges
 * itself (torch.distributed / MPI.Allgather).  Ranks call put / gather the same number of times per buffer. */
typedef struct pgbp_comm pgbp_comm;
int32_t pgbp_comm_create(int32_t device, int32_t rank, int32_t nranks, int64_t ld, int32_t nbuffers,
                         pgbp_comm** out);
int32_t pgbp_comm_handle(pgbp_comm* comm, uint8_t* handle64);
int32_t pgbp_comm_connect(pgbp_comm* comm, const uint8_t* handles /* [nranks][64], rank order */);
/* teardown across processes: every rank disconnects (unmaps its peers), the ranks synchronise, every rank destroys */
int32_t pgbp_comm_disconnect(pgbp_comm* comm);
int32_t pgbp_comm_destroy(pgbp_comm* comm);
/* this rank's window of `buffer`: [nranks][ld] doubles (device pointer) */
int32_t pgbp_comm_window(pgbp_comm* comm, int32_t buffer, double** d_ptr, int64_t* ld);
/* integratebelief!(beliefs, j) for every element, norm[e] written into row `rank` of `buffer` on every rank
 * (enqueue only; src/clustergraphbeliefs.jl:194, src/beliefupdates.jl:168-200) */
int32_t pgbp_integrate_gather(pgbp_batch* batch, int32_t belief, pgbp_comm* comm, int32_t buffer);
/* same exchange for any per-element device vector d_src[B] (e.g. the factored energy of loopy BP) */
int32_t pgbp_comm_put(pgbp_comm* comm, pgbp_batch* batch, int32_t buffer, const double* d_src);
int32_t pgbp_comm_wait(pgbp_comm* comm, pgbp_batch* batch, int32_t buffer, int32_t timeout_ms);
/* host copy of this rank's window of `buffer` ([nranks][ld] doubles); synchronous on the batch's stream */
int32_t pgbp_comm_read(pgbp_comm* comm, pgbp_batch* batch, int32_t buffer, double* host);
/* synchronise the batch's stream and report a wait that timed out (names the missing rank) */
int32_t pgbp_comm_check(pgbp_comm* comm, pgbp_batch* batch);

#ifdef __cplusplus
}
#endif
#endif /* PGBP_B200_H */
